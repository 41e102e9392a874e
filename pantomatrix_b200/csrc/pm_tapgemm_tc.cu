// tcgen05 tap-GEMM: Conv1d (stride 1, any taps / zero padding) and Linear on the Blackwell tensor cores.
//
//   out[b,l,n] = act( bias[n] + sum_t sum_c A[b, l+t-pad, c] * W[t,n,c] + residual[b,l,n] )
//
// Operands are split-bf16 planes (x ~ p0 + p1 + p2, each plane bf16): nsplit 1 = plain bf16, 2 = bf16x3
// (p0*p0 + p0*p1 + p1*p0), 3 = bf16x6 (every product down to 2^-24): all products accumulate in one fp32
// TMEM accumulator, so the result has fp32-grade accuracy at tensor-core rates.
//
// Structure (one 128 x BN output tile per CTA, 320 threads):
//   warp 0   TMA producer  - cp.async.bulk.tensor: A box (64 ch x R rows x NB clips) per plane, with the tap
//                            shift folded into the row coordinate (im2col-free; padding rows are TMA zero fill),
//                            W box (64 ch x BN rows) per plane; 128B-swizzled K-major smem tiles; mbarrier ring
//   warp 1   MMA issuer    - one elected lane issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16),
//                            tcgen05.commit releases smem stages / publishes the accumulator; owns TMEM alloc
//   warps 2-9 epilogue     - tcgen05.ld (32 lanes x 32 columns) -> smem transpose -> bias / residual /
//                            activation -> coalesced fp32 store and/or bf16 split planes for the next GEMM
// Contract and reference call sites: include/pm_emage.h (pm_tapgemm_tc).
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>

#include <cstring>
#include "pm_common.cuh"
#include "../../include/pm_emage.h"


namespace {

constexpr int BM = 128;             // tile rows (UMMA M)
constexpr int BK = 64;              // bf16 channels per k-block = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int A_TILE_BYTES = BM * BK * 2;           // 16 KB per plane
constexpr int NUM_THREADS = 320;   // TMA warp, MMA warp, 8 epilogue warps
constexpr int MAX_STAGES = 8;
constexpr int OCC2_SMEM_KB = 100;   // operand ring per CTA when two CTAs share an SM (2 x (100 + 1.2) KB < 227 KB)
constexpr int HALO_ROWS = 144;      // halo mode: 128 output rows + up to 16 neighbours, whole 8-row swizzle groups
constexpr int HALO_BYTES = HALO_ROWS * BK * 2;      // 18 KB per plane

struct TcParams {
  int taps, pad, nsplit, kblocks;   // kblocks = ceil(cin / 64)
  int rows_out, cout, batch;
  int R, NB;                        // tile = NB clips x R rows (R * NB == 128)
  int w_rows;                       // rows per tap in the packed weight tensor (>= cout, multiple of BN)
  const float* bias;
  const float* residual; long long r_bs; int ldr;
  int act, act_cols; float slope;
  float* out_f32; long long o_bs; int ldo;
  __nv_bfloat16* out_bf16; long long ob_ps, ob_bs; int ldob; int out_nsplit;
  int stages;
  const uint8_t* prefetch; long long prefetch_bytes;   // next GEMM's weights: pulled into L2 while this one runs
  float acc_scale;   // fp16 operands: weights are packed scaled by a power of two, undone here (1 for bf16)
  // ragged batches (pm_tapgemm_tc_rl, nullable): row_limit[clip] valid output rows per clip; the clip of output row
  // (b, l) is b, or (b * rows_out + l) / rows_per_clip when rows_per_clip > 0 (a Linear over all clips as one matrix)
  const int* row_limit; int rows_per_clip;
};

// Instrumented build only (-DPM_TC_TIMING, tools/gemm_timeline.py): per-CTA clock64 stamps of the kernel's phases.
#ifdef PM_TC_TIMING
__device__ unsigned long long pm_tc_stamps[4096 * 8];
#define PM_STAMP(i)                                                                                              \
  do {                                                                                                           \
    if ((threadIdx.x & 31) == 0) {                                                                               \
      const unsigned cta_ = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;                      \
      if (cta_ < 4096) pm_tc_stamps[cta_ * 8 + (i)] = (unsigned long long)clock64();                             \
    }                                                                                                            \
  } while (0)
#else
#define PM_STAMP(i) do {} while (0)
#endif

#include "pm_tc_ptx.cuh"   // PTX wrappers: mbarrier, TMA, tcgen05

// ---------------------------------------------------------------------------------------------------
// CG2 = the CTA-pair form (tcgen05 cta_group::2): two CTAs of a 2-CTA cluster, neighbours along the row-tile axis, work
// on one 256 x BN tile.  Each keeps its own 128 rows of A and its 128 x BN accumulators, but only HALF of the W tile
// (BN / 2 weight rows); the leader's MMAs (M = 256) read both halves.  Why: with two fp16 planes a k-block brings
// 64 KB into shared memory for 12 MMAs of 64 cycles - 83 B / cycle against the ~64 B / cycle an SM can take in from
// L2, so the single-CTA mainloop is fill-bound (1 058 cycles per k-block instead of 768, profiles/r2/gemm_timeline_fp16.txt);
// the pair needs 48 KB per CTA and k-block.
//
// OCC = CTAs per SM the kernel is compiled for.  2 (64-column tiles only: 256 TMEM columns, 96 registers, half the operand
// ring) is for launches of many short tiles - the WavEncoder's 64-channel convs: 7 552 tiles of 15 k-blocks, where one
// resident CTA spent more time in prologue, pipeline fill and epilogue than in its mainloop (13 us per tile against
// 5.7 us of operand fill, profiles/r2/launches_fp16x3.md); with two, one CTA's epilogue overlaps the other's mainloop.
//
// HALO = one-k-block convs (cin <= 64) with several taps.  The tap-GEMM above re-stages the A tile for every tap although
// consecutive taps read the same rows shifted by one: 15 x 32 KB of shared-memory fill per tile of the WavEncoder's
// k = 15 convs, which made them fill-bound.  In halo mode the 128 + taps - 1 input rows of the tile are staged ONCE per
// plane and tap t reads them through a descriptor whose start address is advanced by t rows (t x 128 B).  Measured on
// B200 (profiles/r2/halo_mode_trial.md): the tensor core derives the 128B-swizzle phase from the ADDRESS bits 7-9, so a
// start address that is not 1024-byte aligned needs nothing else - the descriptor's base-offset field must stay 0 (with
// (start >> 7) & 7 in it, as the PTX text suggests for unaligned starts, every result was wrong).  Only the 8 KB W tiles
// stream through the ring.  WavEncoder 64 -> 64, k = 15 conv over 0.97 M rows: 444 -> 420 us.
// Ragged batches: 0 = output row (b, l) is computed as usual, 1 = it lies beyond its clip's row limit and is stored as 0,
// 2 = not stored (outside the output, or a negative limit).  Out of line with scalar arguments: inlined into the
// two-CTAs-per-SM kernels it raised their register spills; this way they spill less than the plain kernels.
__device__ __noinline__ int tc_row_limit(const int* __restrict__ row_limit, int rows_per_clip, int batch, int rows_out,
                                         int b, int l) {
  if (b >= batch || l >= rows_out) return 2;
  int clip = b, r = l;
  if (rows_per_clip > 0) {                                         // batch * rows_out < 2^31 (checked on the host)
    const int g = b * rows_out + l;
    clip = g / rows_per_clip;
    r = g - clip * rows_per_clip;
  }
  const int lim = __ldg(row_limit + clip);
  return r < lim ? 0 : (lim < 0 ? 2 : 1);
}

// RL = the kernel reads per-clip row limits (pm_tapgemm_tc_rl); without them it compiles to exactly the plain kernel.
template <int BN, bool F16, bool CG2, int OCC = 1, bool HALO = false, bool RL = false>
__global__ void __launch_bounds__(NUM_THREADS, OCC) tapgemm_tc_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                    const __grid_constant__ CUtensorMap map_w,
                                                                    const TcParams p) {
  constexpr int W_ROWS_CTA = CG2 ? BN / 2 : BN;     // weight rows this CTA stages per k-block and plane
  constexpr int W_TILE_BYTES = W_ROWS_CTA * BK * 2;
  // instruction descriptor: D = f32; A and B format field 1 = bf16, 0 = fp16; K-major A and B; N >> 3; M >> 4
  constexpr uint32_t IDESC = (1u << 4) | (F16 ? 0u : ((1u << 7) | (1u << 10))) | ((uint32_t)(BN >> 3) << 17) |
                             ((uint32_t)((CG2 ? 2 * BM : BM) >> 4) << 24);
  // Three fp32 accumulators in TMEM: two "main" ones that take the p0*p0 products of alternate k-iterations
  // and one "correction" accumulator for every cross product.  The tensor core aligns and TRUNCATES addends to
  // the accumulator's exponent on every MMA, a biased error ~2^-25 |acc| per instruction; keeping the 2^-8-scaled
  // cross terms apart and halving the chain length of the main sums brings the result back to fp32-FMA quality.
  // The epilogue adds the three in fp32.
  constexpr int TMEM_COLS = BN == 64 ? 256 : 512;   // 3 accumulators rounded up to a power of two
  constexpr int ACC = BN;                           // column stride between the accumulators

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve: [stages][nsplit A tiles][nsplit W tiles] (1024-aligned), then barriers
  uint8_t* tiles = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // halo mode: [nsplit A halo planes][stages][nsplit W tiles]
  const int stage_bytes = HALO ? p.nsplit * W_TILE_BYTES : p.nsplit * (A_TILE_BYTES + W_TILE_BYTES);
  uint8_t* ring = HALO ? tiles + p.nsplit * HALO_BYTES : tiles;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ring + (size_t)p.stages * stage_bytes);
  uint64_t* full_bar = bars;                       // [MAX_STAGES]
  uint64_t* empty_bar = bars + MAX_STAGES;         // [MAX_STAGES]
  uint64_t* acc_bar = bars + 2 * MAX_STAGES;       // accumulator ready
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * MAX_STAGES + 1);
  uint64_t* halo_bar = bars + 2 * MAX_STAGES + 2;  // halo mode: A planes landed

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) PM_STAMP(0);                                   // kernel entry
  const int l0 = blockIdx.x * p.R;
  const int n0 = blockIdx.y * BN;
  const int b0 = blockIdx.z * p.NB;
  const int n_iter = p.taps * p.kblocks;
  const uint32_t cta_rank = CG2 ? cluster_ctarank() : 0u;      // 0 = leader of the pair (issues the MMAs)

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    mbar_init(smem_u32(acc_bar), 1);
    if constexpr (HALO) mbar_init(smem_u32(halo_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if constexpr (CG2) {                                       // one warp of EACH CTA of the pair, same shared-memory slot
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CG2) cluster_sync_all();     // the peer's barriers exist before any remote arrive / TMA completion
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (warp == 0) PM_STAMP(1);                                   // prologue done (barriers, TMEM, descriptors)

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 1 && p.prefetch) {
      // Weights are read once per window and the per-window set (0.6-0.8 GB) does not fit the 126 MB L2, so every
      // GEMM would stream its W tiles from HBM at DRAM latency with only 2-3 stages in flight.  Each CTA instead
      // prefetches its share of the NEXT GEMM's weights into L2 (cp.async.bulk.prefetch.L2) while this one computes.
      const long long ncta = (long long)gridDim.x * gridDim.y * gridDim.z;
      const long long cta = ((long long)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
      long long share = ((p.prefetch_bytes + ncta - 1) / ncta + 127) & ~127LL;
      long long off = cta * share;
      long long end = off + share < p.prefetch_bytes ? off + share : p.prefetch_bytes;
      end &= ~15LL;
      for (; off < end; off += 16384) {
        const uint32_t n = (uint32_t)(end - off < 16384 ? end - off : 16384);
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p.prefetch + off), "r"(n) : "memory");
      }
    }
    if constexpr (HALO) {
      if (elect_one()) {
        mbar_expect_tx(smem_u32(halo_bar), (uint32_t)(p.nsplit * HALO_BYTES));
        for (int pl = 0; pl < p.nsplit; ++pl)
          tma_load_4d(smem_u32(tiles + pl * HALO_BYTES), &map_a, smem_u32(halo_bar), 0, l0 - p.pad, b0, pl);
      }
      __syncwarp();
      int s = 0;
      uint32_t ph = 0;
      for (int it = 0; it < n_iter; ++it) {                      // one W tile pair per tap
        mbar_wait_fast(smem_u32(&empty_bar[s]), ph ^ 1u);
        if (elect_one()) {
          const uint32_t bar = smem_u32(&full_bar[s]);
          mbar_expect_tx(bar, (uint32_t)(p.nsplit * W_TILE_BYTES));
          for (int pl = 0; pl < p.nsplit; ++pl)
            tma_load_3d(smem_u32(ring + (size_t)s * stage_bytes + pl * W_TILE_BYTES), &map_w, bar, 0, it * p.w_rows + n0, pl);
        }
        __syncwarp();
        if (++s == p.stages) { s = 0; ph ^= 1u; }
      }
    } else {
      const uint32_t tx = (uint32_t)(p.nsplit * (A_TILE_BYTES + W_TILE_BYTES));
      int s = 0, tap = 0, kb = 0;
      uint32_t ph = 0;
      for (int it = 0; it < n_iter; ++it) {
        mbar_wait_fast(smem_u32(&empty_bar[s]), ph ^ 1u);       // whole warp waits (uniform control flow)
        const uint32_t bar = smem_u32(&full_bar[s]);
        uint8_t* st = tiles + (size_t)s * stage_bytes;
        if (elect_one()) {
        if constexpr (CG2) {
          // Both CTAs' bytes land on the LEADER's barrier, which expects 2 x tx; the peer's barrier is unused.  (The
          // peer cannot run a phase ahead: it reuses a stage only after the leader's MMAs of the previous use have
          // committed.  A cluster-scope release arrive from the peer per k-block was tried first and serialised the
          // peer's producer: 1 430 cycles per k-block whatever the work.)
          if (cta_rank == 0) mbar_expect_tx(bar, 2 * tx);
        } else {
          mbar_expect_tx(bar, tx);
        }
        for (int pl = 0; pl < p.nsplit; ++pl) {
          const uint32_t a_dst = smem_u32(st + pl * A_TILE_BYTES);
          const uint32_t w_dst = smem_u32(st + p.nsplit * A_TILE_BYTES + pl * W_TILE_BYTES);
          if constexpr (CG2) {
            tma_load_4d_cg2(a_dst, &map_a, bar, kb * BK, l0 + tap - p.pad, b0, pl);
            tma_load_3d_cg2(w_dst, &map_w, bar, kb * BK, tap * p.w_rows + n0 + (int)cta_rank * W_ROWS_CTA, pl);
          } else {
            tma_load_4d(a_dst, &map_a, bar, kb * BK, l0 + tap - p.pad, b0, pl);
            tma_load_3d(w_dst, &map_w, bar, kb * BK, tap * p.w_rows + n0, pl);
          }
        }
        }
        __syncwarp();
        if (++s == p.stages) { s = 0; ph ^= 1u; }
        if (++kb == p.kblocks) { kb = 0; ++tap; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (pair: the leader CTA only; the peer's warp 1 only owns its TMEM allocation) =====
    if (cta_rank == 0)
    // One thread feeds the tensor core, so its own instruction stream must stay far below the 64 cycles a
    // 128x128x16 MMA takes.  Measured: with per-MMA descriptor construction, runtime div/mod for the stage ring
    // and a clock-reading wait loop this thread was THE bottleneck (the mainloop ran at the same speed with all TMA
    // loads disabled, profiles/gemm_microbench_r1.md).  Hence: running stage/phase counters, descriptors advanced by
    // adding to a precomputed 64-bit base, product loops specialised per split mode and fully unrolled.
    {
      const uint64_t desc_hi = (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
      auto mma = [](uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
        if constexpr (CG2) tc_mma_cg2(d, a, b, idesc, acc);
        else tc_mma_bf16(d, a, b, idesc, acc);
      };
      auto commit = [](uint32_t bar) {
        if constexpr (CG2) tc_commit_cg2(bar);               // arrives in both CTAs of the pair
        else tc_commit(bar);
      };
      const uint32_t tiles_u32 = smem_u32(tiles);
      const uint32_t ring_u32 = smem_u32(ring);
      const uint32_t d_corr = tmem_base + 2 * ACC;
      if constexpr (HALO) {
        mbar_wait_fast(smem_u32(halo_bar), 0);
        tc_fence_after();
      }
      uint32_t first_main0 = 1, first_main1 = 1, first_corr = 1;     // 1 until the accumulator has been written once
      int s = 0;
      uint32_t ph = 0;
      for (int it = 0; it < n_iter; ++it) {
        mbar_wait_fast(smem_u32(&full_bar[s]), ph);               // whole warp waits (uniform control flow)
        tc_fence_after();
        if (it == 0) PM_STAMP(2);                                 // first operand stage landed
        if (elect_one()) {
        const uint32_t a_base = HALO ? tiles_u32 + (uint32_t)it * 128u                             // tap = row shift
                                     : tiles_u32 + (uint32_t)s * (uint32_t)stage_bytes;
        const uint32_t w_base = HALO ? ring_u32 + (uint32_t)s * (uint32_t)stage_bytes : a_base + p.nsplit * A_TILE_BYTES;
        // halo: the start address sits (it % 8) rows into a 1024-byte swizzle atom; base offset (bits 49-51) stays 0
        const uint64_t a0 = desc_hi | (uint64_t)((a_base >> 4) & 0x3FFFu);
        const uint64_t w0 = desc_hi | (uint64_t)((w_base >> 4) & 0x3FFFu);
        constexpr uint64_t A_PL = (HALO ? HALO_BYTES : A_TILE_BYTES) >> 4, W_PL = W_TILE_BYTES >> 4, K_ST = (UMMA_K * 2) >> 4;   // descriptor units
        const bool odd = it & 1;
        const uint32_t d_main = tmem_base + (odd ? ACC : 0);
        // cross products first (small -> large), into the correction accumulator
        if (p.nsplit == 3) {
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) mma(d_corr, a0 + k * K_ST, w0 + 2 * W_PL + k * K_ST, IDESC, (k | (int)(first_corr ^ 1u)) != 0);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) mma(d_corr, a0 + A_PL + k * K_ST, w0 + W_PL + k * K_ST, IDESC, 1);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) mma(d_corr, a0 + 2 * A_PL + k * K_ST, w0 + k * K_ST, IDESC, 1);
        }
        if (p.nsplit >= 2) {
          const uint32_t fresh = p.nsplit == 3 ? 0u : first_corr;      // with 3 planes the block above already wrote it
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) mma(d_corr, a0 + k * K_ST, w0 + W_PL + k * K_ST, IDESC, (k | (int)(fresh ^ 1u)) != 0);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) mma(d_corr, a0 + A_PL + k * K_ST, w0 + k * K_ST, IDESC, 1);
        }
        {
          const uint32_t first = odd ? first_main1 : first_main0;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) mma(d_main, a0 + k * K_ST, w0 + k * K_ST, IDESC, (k | (int)(first ^ 1u)) != 0);
        }
        commit(smem_u32(&empty_bar[s]));             // frees this smem stage when the MMAs have read it
        }
        __syncwarp();
        if (p.nsplit >= 2) first_corr = 0;
        if (it & 1) first_main1 = 0; else first_main0 = 0;
        if (++s == p.stages) { s = 0; ph ^= 1u; }
      }
      if (n_iter > 0 && elect_one()) commit(smem_u32(acc_bar));      // accumulator complete
      PM_STAMP(3);                                                // all MMAs issued
    }
  } else {
    // ===== epilogue warps 2..9: TMEM lane quarter = warp % 4, column half = (warp - 2) / 4 =====
    // tcgen05.ld hands each thread one accumulator ROW (32 consecutive columns).  The 32x32 chunk is transposed
    // through shared memory (the operand ring is idle by now) so that each quarter-warp writes one contiguous
    // 128-byte row segment.  Measured (profiles/gemm_microbench_r1.md): with 4 warps and branchy per-element code
    // the epilogue cost 12 us of a 16 us GEMM - it is instruction-latency bound (one warp per scheduler), not
    // memory bound - hence 8 warps, branch-free activation (identity == leaky with slope 1) and a warp-uniform
    // fast path for full chunks.
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    constexpr int CW = 32;                                         // columns per tcgen05.ld chunk
    constexpr int LPR = CW / 4;                                    // lanes per staged row (one float4 each)
    constexpr int RPI = 32 / LPR;                                  // rows written per warp-wide store
    constexpr int NIT = 32 / RPI;                                  // store rounds per chunk
    constexpr int ST = CW + 4;                                     // staging row stride (floats): 16B aligned, conflict-free
    const uint32_t stage = smem_u32(tiles) + (warp - 2) * 32 * ST * 4;   // <= 4.6 KB per warp (shared-space address)
    const int sub_r = lane / LPR, c4 = (lane % LPR) * 4;           // this lane's row-in-group / first column of its float4
    const int r_shift = 31 - __clz(p.R);                           // R is a power of two
    const bool vec_f = p.out_f32 && ((p.ldo & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.out_f32) & 15) == 0) && ((p.o_bs & 3) == 0);
    const bool vec_r = p.residual && ((p.ldr & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.residual) & 15) == 0) && ((p.r_bs & 3) == 0);
    const bool vec_b = p.out_bf16 && ((p.ldob & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.out_bf16) & 7) == 0) &&
                       ((p.ob_bs & 3) == 0) && ((p.ob_ps & 3) == 0);
    const bool all_vec = (!p.out_f32 || vec_f) && (!p.residual || vec_r) && (!p.out_bf16 || vec_b);
    const float act_slope = p.act == PM_ACT_NONE ? 1.f : (p.act == PM_ACT_RELU ? 0.f : p.slope);
    // rows this lane stores (NIT per chunk): offsets are chunk-invariant
    long long off_f[NIT], off_r[NIT], off_b[NIT];
    uint32_t row_ok = 0;
#pragma unroll
    for (int i = 0; i < NIT; ++i) {
      const int rt = q * 32 + RPI * i + sub_r;
      const int b = b0 + (rt >> r_shift), l = l0 + (rt & (p.R - 1));
      if (b < p.batch && l < p.rows_out) row_ok |= 1u << i;
      off_f[i] = (long long)b * p.o_bs + (long long)l * p.ldo;
      off_r[i] = (long long)b * p.r_bs + (long long)l * p.ldr;
      off_b[i] = (long long)b * p.ob_bs + (long long)l * p.ldob;
    }
    // Ragged batch: rows beyond their clip's limit leave the computed set here and are zeroed after the chunk loop,
    // so the hot loop below is the same code with or without limits (rolled, recomputed: no registers held across it).
    if (RL && p.row_limit) {
#pragma unroll 1
      for (int i = 0; i < NIT; ++i)
        if (tc_row_limit(p.row_limit, p.rows_per_clip, p.batch, p.rows_out, b0 + ((q * 32 + RPI * i + sub_r) >> r_shift),
                         l0 + ((q * 32 + RPI * i + sub_r) & (p.R - 1))) != 0)
          row_ok &= ~(1u << i);
    }
#pragma unroll 1
    for (int c0 = half * (BN / 2); c0 < (half + 1) * (BN / 2); c0 += CW) {
      uint32_t acc[CW];
      float v[CW];
      const uint32_t lane_col = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;
      // Everything that does not depend on the accumulators - row offsets above, this chunk's bias and residual
      // loads - is issued BEFORE the accumulator wait / TMEM loads, so their global latency overlaps the tail of the
      // mainloop instead of sitting in the epilogue (measured round 2: 33.4 -> 30.6 ms per step in bf16x6 mode,
      // 26.5 -> 23.9 ms in fp16x3, profiles/README.md).
      const int nb = n0 + c0;                                                      // first column of this chunk
      const int n = nb + c4;                                                       // this lane's first column
      const bool fast = all_vec && nb + CW <= p.cout;                              // warp-uniform: whole chunk inside cout
      float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p.bias) {
        if (n < p.cout) bias4.x = __ldg(p.bias + n);
        if (n + 1 < p.cout) bias4.y = __ldg(p.bias + n + 1);
        if (n + 2 < p.cout) bias4.z = __ldg(p.bias + n + 2);
        if (n + 3 < p.cout) bias4.w = __ldg(p.bias + n + 3);
      }
      float4 rres[NIT];
      if (fast && p.residual) {
#pragma unroll
        for (int i = 0; i < NIT; ++i)
          rres[i] = ((row_ok >> i) & 1u) ? *reinterpret_cast<const float4*>(p.residual + off_r[i] + n) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      if (c0 == half * (BN / 2)) {
        mbar_wait(smem_u32(acc_bar), 0);
        tc_fence_after();
        if (warp == 2) PM_STAMP(4);                                 // accumulators complete
      }
      __syncwarp();                                                                // .sync.aligned: whole warp converged
      tmem_ld(lane_col, acc);
#pragma unroll
      for (int j = 0; j < CW; ++j) v[j] = __uint_as_float(acc[j]);
      if (n_iter > 1) {                                                            // second main accumulator in use
        tmem_ld(lane_col + ACC, acc);
#pragma unroll
        for (int j = 0; j < CW; ++j) v[j] += __uint_as_float(acc[j]);
      }
      if (p.nsplit > 1) {                                                          // cross-product accumulator
        tmem_ld(lane_col + 2 * ACC, acc);
#pragma unroll
        for (int j = 0; j < CW; ++j) v[j] += __uint_as_float(acc[j]);
      }
      if constexpr (F16) {                                                         // undo the weight pre-scale (exact)
#pragma unroll
        for (int j = 0; j < CW; ++j) v[j] *= p.acc_scale;
      }
      if (nb >= p.cout) continue;                                   // warp-uniform
      // transpose: thread = row -> smem[row][0..CW)
#pragma unroll
      for (int j = 0; j < CW / 4; ++j) sts128(stage + (lane * ST + 4 * j) * 4, v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      __syncwarp();
      // identity == leaky with slope 1: one branch-free (select) formula for none / relu / leaky / partial activation
      const float s0 = n < p.act_cols ? act_slope : 1.f, s1 = n + 1 < p.act_cols ? act_slope : 1.f;
      const float s2 = n + 2 < p.act_cols ? act_slope : 1.f, s3 = n + 3 < p.act_cols ? act_slope : 1.f;
      if (fast) {
        // Hot path, kept contiguous and small: the ragged path below is rolled and placed after it, so the
        // instructions actually executed do not straddle 200+ KB of cold unrolled code (in-kernel clock stamps,
        // profiles/gemm_timeline_r1.txt: the epilogue was instruction-fetch bound).
#pragma unroll
        for (int i = 0; i < NIT; ++i) {
          if (!((row_ok >> i) & 1u)) continue;
          float4 x = lds128(stage + ((RPI * i + sub_r) * ST + c4) * 4);
          x.x += bias4.x; x.y += bias4.y; x.z += bias4.z; x.w += bias4.w;
          if (p.residual) {
            const float4 t = rres[i];
            x.x += t.x; x.y += t.y; x.z += t.z; x.w += t.w;
          }
          // compare-select, not fmaxf / fminf: those return the non-NaN operand and would turn the NaN an fp16 operand
          // overflow leaves into 0, hiding it from the overflow guard (round 2: a 2e4x too loud input went unnoticed)
          x.x = x.x < 0.f ? s0 * x.x : x.x;
          x.y = x.y < 0.f ? s1 * x.y : x.y;
          x.z = x.z < 0.f ? s2 * x.z : x.z;
          x.w = x.w < 0.f ? s3 * x.w : x.w;
          if (p.out_f32) *reinterpret_cast<float4*>(p.out_f32 + off_f[i] + n) = x;
          if (p.out_bf16) {
            const PmPlanes P{p.out_bf16 + off_b[i], p.ob_ps, p.ldob, p.out_nsplit};
            pm_store_planes4_t<F16>(P, 0, n, x);
          }
        }
      } else if (n < p.cout) {
        // ragged / unaligned tail: per element, rolled (offsets recomputed so the arrays above stay in registers)
#pragma unroll 1
        for (int i = 0; i < NIT; ++i) {
          const int rt = q * 32 + RPI * i + sub_r;
          const int b = b0 + (rt >> r_shift), l = l0 + (rt & (p.R - 1));
          if (RL ? !((row_ok >> i) & 1u) : (b >= p.batch || l >= p.rows_out)) continue;
          const long long of = (long long)b * p.o_bs + (long long)l * p.ldo;
          const long long orr = (long long)b * p.r_bs + (long long)l * p.ldr;
          const PmPlanes P{p.out_bf16 ? p.out_bf16 + (long long)b * p.ob_bs + (long long)l * p.ldob : nullptr,
                           p.ob_ps, p.ldob, p.out_nsplit};
          const uint32_t src = stage + ((RPI * i + sub_r) * ST + c4) * 4;
#pragma unroll 1
          for (int k = 0; k < 4; ++k) {
            if (n + k >= p.cout) break;
            float y;
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(y) : "r"(src + 4 * k) : "memory");
            y += k == 0 ? bias4.x : (k == 1 ? bias4.y : (k == 2 ? bias4.z : bias4.w));
            if (p.residual) y += p.residual[orr + n + k];
            y = y < 0.f ? (k == 0 ? s0 : (k == 1 ? s1 : (k == 2 ? s2 : s3))) * y : y;
            if (p.out_f32) p.out_f32[of + n + k] = y;
            if (P.ptr) pm_store_planes_t<F16>(P, 0, n + k, y);
          }
        }
      }
    }
  }
  // Ragged batch: the rows of this CTA beyond their clip's limit, stored as 0 by all 8 epilogue warps (after the
  // epilogue proper, with nothing it holds in registers: the hot epilogue is the same code with or without limits).
  if (RL && p.row_limit && warp >= 2) {
#pragma unroll 1
    for (int rt = warp - 2; rt < BM; rt += 8) {
      const int b = blockIdx.z * p.NB + rt / p.R, l = blockIdx.x * p.R + rt % p.R;
      if (tc_row_limit(p.row_limit, p.rows_per_clip, p.batch, p.rows_out, b, l) != 1) continue;
      const PmPlanes P{p.out_bf16 ? p.out_bf16 + (long long)b * p.ob_bs + (long long)l * p.ldob : nullptr,
                       p.ob_ps, p.ldob, p.out_nsplit};
#pragma unroll 1
      for (int n = blockIdx.y * BN + lane; n < blockIdx.y * BN + BN && n < p.cout; n += 32) {
        if (p.out_f32) p.out_f32[(long long)b * p.o_bs + (long long)l * p.ldo + n] = 0.f;
        if (P.ptr) pm_store_planes_t<F16>(P, 0, n, 0.f);
      }
    }
  }

  if (warp == 2) PM_STAMP(5);                                     // this warp's share of the epilogue issued
  // teardown: everyone done with TMEM before the owning warp frees it
  tc_fence_before();
  __syncthreads();
  if (warp == 0) PM_STAMP(6);                                     // all warps done
  if constexpr (CG2) cluster_sync_all();    // neither CTA frees TMEM or leaves while the peer may still signal its barriers
  if (warp == 1) {
    tc_fence_after();
    if constexpr (CG2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------
// fp32 -> bf16 planes.  One CTA row-block per (clip, row tile): no per-element index arithmetic, 16-byte loads,
// 8-byte stores.  VEC path needs ch % 4 == 0 and 16-byte aligned rows.
template <bool VEC, bool F16>
__global__ void __launch_bounds__(256) split_bf16_kernel(const float* __restrict__ x, long long x_bs, int ldx, int rows,
                                                         int ch, __nv_bfloat16* __restrict__ out, long long o_ps,
                                                         long long o_bs, int ldo, int nsplit) {
  const int b = blockIdx.y;
  const float* __restrict__ xb = x + (long long)b * x_bs;
  __nv_bfloat16* __restrict__ ob = out + (long long)b * o_bs;
  if (VEC) {
    const int ch4 = ch >> 2;
    const long long total = (long long)rows * ch4;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const int r = (int)(i / ch4), c4 = (int)(i - (long long)r * ch4);
      const float4 v = *reinterpret_cast<const float4*>(xb + (long long)r * ldx + 4 * c4);
      const PmPlanes P{ob, o_ps, ldo, nsplit};
      pm_store_planes4_t<F16>(P, r, 4 * c4, v);
    }
  } else {
    const long long total = (long long)rows * ch;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const int r = (int)(i / ch), c = (int)(i - (long long)r * ch);
      const PmPlanes P{ob, o_ps, ldo, nsplit};
      pm_store_planes_t<F16>(P, r, c, xb[(long long)r * ldx + c]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
template <int BN, bool F16, bool CG2, int OCC = 1, bool HALO = false, bool RL = false>
int launch(const CUtensorMap& ma, const CUtensorMap& mw, TcParams& p, dim3 grid, cudaStream_t st, int pair_axis = 0) {
  static_assert(OCC == 1 || (BN == 64 && !CG2), "two CTAs per SM: 64-column tiles only (TMEM columns, registers)");
  static_assert(!HALO || (OCC == 2 && BN == 64), "halo mode is built for the 64-column, two-CTAs-per-SM form");
  const int stage_bytes = HALO ? p.nsplit * BN * BK * 2 : p.nsplit * (A_TILE_BYTES + (CG2 ? BN / 2 : BN) * BK * 2);
  const int fixed_bytes = HALO ? p.nsplit * HALO_BYTES : 0;
  static const int env_kb = getenv("PM_TC_SMEM_KB") ? atoi(getenv("PM_TC_SMEM_KB")) : 200;   // tuning override
  int stages = ((OCC == 2 ? OCC2_SMEM_KB : env_kb) * 1024 - fixed_bytes) / stage_bytes;
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  if (stages < 2) return PM_EUNSUPPORTED;
  p.stages = stages;
  const size_t smem = (size_t)fixed_bytes + (size_t)stages * stage_bytes + 1024 /*align slack*/ + (2 * MAX_STAGES + 3) * sizeof(uint64_t);
  static unsigned long long configured = 0;       // per template instantiation, one bit per device
  if (pm_first_use_on_device(configured)) {
    cudaError_t e = cudaFuncSetAttribute(tapgemm_tc_kernel<BN, F16, CG2, OCC, HALO, RL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) { configured = 0; return (int)e; }
  }
  if constexpr (CG2) {                      // CTA pairs: 2-CTA clusters along the row-tile axis
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = pair_axis == 0 ? 2 : 1;       // the pair: two row tiles (x) or two clip tiles (z) of one N tile
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = pair_axis == 2 ? 2 : 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, tapgemm_tc_kernel<BN, F16, CG2, OCC, HALO, RL>, ma, mw, p);
    return e == cudaSuccess ? PM_OK : (int)e;
  } else {
    tapgemm_tc_kernel<BN, F16, CG2, OCC, HALO, RL><<<grid, NUM_THREADS, smem, st>>>(ma, mw, p);
    PM_LAUNCH_CHECK();
  }
}

template <bool RL>
int dispatch(const CUtensorMap& ma, const CUtensorMap& mw, TcParams& p, dim3 grid, cudaStream_t st, bool halo, bool f16,
             bool cg2, bool occ2, int BNsel, int pair_axis) {
  if (halo) {
    if (f16) return launch<64, true, false, 2, true, RL>(ma, mw, p, grid, st);
    return launch<64, false, false, 2, true, RL>(ma, mw, p, grid, st);
  }
  if (f16) {
    if (cg2) return launch<128, true, true, 1, false, RL>(ma, mw, p, grid, st, pair_axis);
    if (occ2) return launch<64, true, false, 2, false, RL>(ma, mw, p, grid, st);
    if (BNsel == 64) return launch<64, true, false, 1, false, RL>(ma, mw, p, grid, st);
    return launch<128, true, false, 1, false, RL>(ma, mw, p, grid, st);
  }
  if (occ2) return launch<64, false, false, 2, false, RL>(ma, mw, p, grid, st);
  if (BNsel == 64) return launch<64, false, false, 1, false, RL>(ma, mw, p, grid, st);
  return launch<128, false, false, 1, false, RL>(ma, mw, p, grid, st);
}

}  // namespace

static int tapgemm_tc_run(const uint16_t* A, long long a_ps, long long a_bs, int lda, int batch, int rows_in, int cin,
                          const uint16_t* W, long long w_ps, int w_rows, int ldw, int taps, int pad, int nsplit,
                          const float* bias, int rows_out, int cout,
                          const float* residual, long long r_bs, int ldr,
                          int act, int act_cols, float slope, float acc_scale,
                          float* out_f32, long long o_bs, int ldo,
                          uint16_t* out_bf16, long long ob_ps, long long ob_bs, int ldob, int out_nsplit,
                          const void* prefetch, long long prefetch_bytes, const int* row_limit, int rows_per_clip,
                          void* stream) {
  PM_REQUIRE(A && W && (out_f32 || out_bf16));
  PM_TAKE_FMT(nsplit, f16);                 // operand planes: bf16 (default) or fp16
  PM_TAKE_FMT(out_nsplit, out_f16);
  PM_REQUIRE(!out_bf16 || out_f16 == f16);  // emitted planes use the operand format
  PM_REQUIRE(f16 || acc_scale == 1.0f);
  PM_REQUIRE(!prefetch || (prefetch_bytes >= 0 && (reinterpret_cast<uintptr_t>(prefetch) & 15) == 0));
  PM_REQUIRE(batch > 0 && rows_in > 0 && rows_out > 0 && cin > 0 && cout > 0 && taps > 0);
  PM_REQUIRE(nsplit >= 1 && nsplit <= 3 && (!out_bf16 || (out_nsplit >= 1 && out_nsplit <= 3)));
  PM_REQUIRE(act >= PM_ACT_NONE && act <= PM_ACT_LEAKY);
  // TMA: 16-byte aligned base and strides
  PM_REQUIRE((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0);
  PM_REQUIRE((lda & 7) == 0 && (ldw & 7) == 0 && lda >= cin && ldw >= cin && w_rows >= cout);
  PM_REQUIRE(batch == 1 || (a_bs & 7) == 0);
  PM_REQUIRE(nsplit == 1 || ((a_ps & 7) == 0 && (w_ps & 7) == 0));
  PM_REQUIRE(!out_f32 || ldo >= cout);
  PM_REQUIRE(!out_bf16 || ldob >= cout);
  PM_REQUIRE(!residual || ldr >= cout);

  int R = 128;
  if (rows_out <= 64 && batch > 1) { R = 16; while (R < rows_out) R <<= 1; }
  const int NB = 128 / R;
  // N tile: 128 columns (64 for narrow outputs).  Measured alternatives that lost and were removed: 64-column tiles for
  // the M = 2048 GEMMs, 96-column tiles (34.2 vs 33.4 ms per step), 2x2 clusters with TMA multicast (10-25 % slower),
  // programmatic dependent launch (35.2 vs 34.7 ms): profiles/README.md.
  int BNsel = cout <= 64 ? 64 : 128;
  PM_REQUIRE(w_rows % BNsel == 0);
  // CTA pairs (cta_group::2) where the row-tile grid is even: two fp16 planes, 128-column tiles, 128-row tiles.
  static const bool cg2_on = !(getenv("PM_TC_CG2") && atoi(getenv("PM_TC_CG2")) == 0);      // A/B switch (tools)
  // Measured (profiles/r2/gemm_microbench_fp16_pairs.txt, M = 2048, N = 768): K = 768 12.4 vs 13.5 us, K = 1536 18.1 vs
  // 20.8, K = 3072 29.0 vs 35.5 (906 instead of 1 184 cycles per k-block: MMA-bound); K <= 256 is a few hundred ns
  // slower (cluster barriers in prologue and teardown), hence the k-block threshold.
  // Pairs are formed along the row-tile axis only.  (Pairing clip tiles of the batch-tiled small-R convs along z was
  // tried and failed the golden parity tests on the first run; it was not pursued - those convs are a few per cent
  // of the step.)
  const int pair_axis = 0;
  const bool cg2 = cg2_on && f16 && nsplit == 2 && BNsel == 128 && R == 128 && pm_cdiv(rows_out, R) % 2 == 0 &&
                   taps * ((cin + BK - 1) / BK) >= 6;

  // Halo mode (see the kernel): one-k-block convs with >= 3 taps on 128-row tiles, two fp16 / bf16 planes.
  static const bool halo_on = !(getenv("PM_TC_HALO") && atoi(getenv("PM_TC_HALO")) == 0);      // A/B switch (tools)
  const bool halo = halo_on && BNsel == 64 && R == 128 && cin <= BK && taps >= 3 && BM + taps - 1 <= HALO_ROWS && nsplit == 2;

  TcParams p;
  p.taps = taps; p.pad = pad; p.nsplit = nsplit; p.kblocks = (cin + BK - 1) / BK;
  p.rows_out = rows_out; p.cout = cout; p.batch = batch; p.R = R; p.NB = NB; p.w_rows = w_rows;
  p.bias = bias; p.residual = residual; p.r_bs = r_bs; p.ldr = ldr;
  p.act = act; p.act_cols = act_cols <= 0 ? cout : act_cols; p.slope = slope;
  p.out_f32 = out_f32; p.o_bs = o_bs; p.ldo = ldo;
  p.out_bf16 = reinterpret_cast<__nv_bfloat16*>(out_bf16); p.ob_ps = ob_ps; p.ob_bs = ob_bs; p.ldob = ldob;
  p.out_nsplit = out_bf16 ? out_nsplit : 0;
  p.stages = 0;
  p.prefetch = static_cast<const uint8_t*>(prefetch);
  p.prefetch_bytes = prefetch ? prefetch_bytes : 0;
  p.acc_scale = acc_scale;
  p.row_limit = row_limit; p.rows_per_clip = rows_per_clip;
  CUtensorMap ma, mw;
  {
    const long long bs_el = batch > 1 ? a_bs : (long long)rows_in * lda;
    const long long ps_el = nsplit > 1 ? a_ps : bs_el * batch;
    cuuint64_t dims[4] = {(cuuint64_t)cin, (cuuint64_t)rows_in, (cuuint64_t)batch, (cuuint64_t)nsplit};
    cuuint64_t strides[3] = {(cuuint64_t)lda * 2, (cuuint64_t)bs_el * 2, (cuuint64_t)ps_el * 2};
    cuuint32_t box[4] = {(cuuint32_t)BK, (cuuint32_t)(halo ? HALO_ROWS : R), (cuuint32_t)NB, 1};
    if (!encode_map(&ma, A, 4, dims, strides, box, f16)) return PM_EBADARG;
  }
  {
    const long long ps_el = nsplit > 1 ? w_ps : (long long)taps * w_rows * ldw;
    cuuint64_t dims[3] = {(cuuint64_t)cin, (cuuint64_t)taps * w_rows, (cuuint64_t)nsplit};
    cuuint64_t strides[2] = {(cuuint64_t)ldw * 2, (cuuint64_t)ps_el * 2};
    cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)(cg2 ? BNsel / 2 : BNsel), 1};      // pair: each CTA stages half of the W tile
    if (!encode_map(&mw, W, 3, dims, strides, box, f16)) return PM_EBADARG;
  }
  dim3 grid(pm_cdiv(rows_out, R), pm_cdiv(cout, BNsel), pm_cdiv(batch, NB));
  PM_REQUIRE(grid.z <= 65535 && grid.y <= 65535);
  // Two CTAs per SM for 64-column launches with more tiles than two per SM, if half the ring still holds 2 stages.
  static const bool occ2_on = !(getenv("PM_TC_OCC2") && atoi(getenv("PM_TC_OCC2")) == 0);      // A/B switch (tools)
  const bool occ2 = occ2_on && BNsel == 64 && (long long)grid.x * grid.y * grid.z > 2 * 148 &&
                    OCC2_SMEM_KB * 1024 / (nsplit * (A_TILE_BYTES + 64 * BK * 2)) >= 2;
  if (row_limit) return dispatch<true>(ma, mw, p, grid, (cudaStream_t)stream, halo, f16, cg2, occ2, BNsel, pair_axis);
  return dispatch<false>(ma, mw, p, grid, (cudaStream_t)stream, halo, f16, cg2, occ2, BNsel, pair_axis);
}

extern "C" int pm_tapgemm_tc(const uint16_t* A, long long a_ps, long long a_bs, int lda, int batch, int rows_in, int cin,
                             const uint16_t* W, long long w_ps, int w_rows, int ldw, int taps, int pad, int nsplit,
                             const float* bias, int rows_out, int cout,
                             const float* residual, long long r_bs, int ldr,
                             int act, int act_cols, float slope, float acc_scale,
                             float* out_f32, long long o_bs, int ldo,
                             uint16_t* out_bf16, long long ob_ps, long long ob_bs, int ldob, int out_nsplit,
                             const void* prefetch, long long prefetch_bytes, void* stream) {
  return tapgemm_tc_run(A, a_ps, a_bs, lda, batch, rows_in, cin, W, w_ps, w_rows, ldw, taps, pad, nsplit, bias, rows_out,
                        cout, residual, r_bs, ldr, act, act_cols, slope, acc_scale, out_f32, o_bs, ldo, out_bf16, ob_ps,
                        ob_bs, ldob, out_nsplit, prefetch, prefetch_bytes, nullptr, 0, stream);
}

extern "C" int pm_tapgemm_tc_rl(const uint16_t* A, long long a_ps, long long a_bs, int lda, int batch, int rows_in, int cin,
                                const uint16_t* W, long long w_ps, int w_rows, int ldw, int taps, int pad, int nsplit,
                                const float* bias, int rows_out, int cout,
                                const float* residual, long long r_bs, int ldr,
                                int act, int act_cols, float slope, float acc_scale,
                                float* out_f32, long long o_bs, int ldo,
                                uint16_t* out_bf16, long long ob_ps, long long ob_bs, int ldob, int out_nsplit,
                                const void* prefetch, long long prefetch_bytes, const int* row_limit, int rows_per_clip,
                                void* stream) {
  PM_REQUIRE(rows_per_clip >= 0 && (long long)batch * rows_out < (1LL << 31));
  return tapgemm_tc_run(A, a_ps, a_bs, lda, batch, rows_in, cin, W, w_ps, w_rows, ldw, taps, pad, nsplit, bias, rows_out,
                        cout, residual, r_bs, ldr, act, act_cols, slope, acc_scale, out_f32, o_bs, ldo, out_bf16, ob_ps,
                        ob_bs, ldob, out_nsplit, prefetch, prefetch_bytes, row_limit, rows_per_clip, stream);
}

#ifdef PM_TC_TIMING
extern "C" int pm_tc_timing_reset() {
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return (int)e;
  void* d = nullptr;
  e = cudaGetSymbolAddress(&d, pm_tc_stamps);
  if (e != cudaSuccess) return (int)e;
  return (int)cudaMemset(d, 0, sizeof(unsigned long long) * 4096 * 8);
}
extern "C" int pm_tc_timing_read(unsigned long long* host) {
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return (int)e;
  return (int)cudaMemcpyFromSymbol(host, pm_tc_stamps, sizeof(unsigned long long) * 4096 * 8);
}
#endif

extern "C" int pm_split_bf16(const float* x, long long x_bs, int ldx, int batch, int rows, int ch,
                             uint16_t* out, long long o_ps, long long o_bs, int ldo, int nsplit, void* stream) {
  PM_TAKE_FMT(nsplit, f16);
  PM_REQUIRE(x && out && batch >= 0 && rows >= 0 && ch > 0 && ldx >= ch && ldo >= ch && nsplit >= 1 && nsplit <= 3);
  if ((long long)batch * rows == 0) return PM_OK;
  PM_REQUIRE(batch <= 65535);
  const bool vec = (ch & 3) == 0 && (ldx & 3) == 0 && (x_bs & 3) == 0 && (ldo & 3) == 0 && (o_bs & 3) == 0 &&
                   (o_ps & 3) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 7) == 0;
  const long long work = (long long)rows * (vec ? ch / 4 : ch);
  long long gx = (work + 255) / 256;
  const long long cap = batch >= 148 * 4 ? 1 : (148 * 8 + batch - 1) / batch;
  if (gx > cap) gx = cap;
  dim3 grid((unsigned)gx, batch);
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
  cudaStream_t st = (cudaStream_t)stream;
  if (f16) {
    if (vec) split_bf16_kernel<true, true><<<grid, 256, 0, st>>>(x, x_bs, ldx, rows, ch, o, o_ps, o_bs, ldo, nsplit);
    else split_bf16_kernel<false, true><<<grid, 256, 0, st>>>(x, x_bs, ldx, rows, ch, o, o_ps, o_bs, ldo, nsplit);
  } else {
    if (vec) split_bf16_kernel<true, false><<<grid, 256, 0, st>>>(x, x_bs, ldx, rows, ch, o, o_ps, o_bs, ldo, nsplit);
    else split_bf16_kernel<false, false><<<grid, 256, 0, st>>>(x, x_bs, ldx, rows, ch, o, o_ps, o_bs, ldo, nsplit);
  }
  PM_LAUNCH_CHECK();
}
