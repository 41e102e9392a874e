// Multi-head attention core on the tcgen05 tensor cores (T <= 64 tokens, head_dim 192, no masks): the whole
// 64 x 64 score tile of one (clip, head) lives in TMEM, softmax runs in registers, P goes back through shared
// memory as the A operand of the P.V product.  Contract: include/pm_emage.h (pm_attention_tc); replaces
// scaled_dot_product_attention inside nn.MultiheadAttention of every transformer layer (M.py:238-250).
//
// Operands are the two-plane fp16 activations of the fp16x3 engine (x = (p0 + p1) / 64, pm_common.cuh), written
// by the producing GEMM's epilogue, so Q, K, V arrive by TMA straight from the packed q|k|v projection output:
//   S  = Q K^T            3 products (p0 p0 + p0 p1 + p1 p0), UMMA M=64 N=64 K=16, A and B K-major (dims contiguous)
//   P  = exp(S/sqrt(hd) - rowmax)   fp32 in registers (thread = query row), split into two fp16 planes of 1024 P
//   O  = P V              3 products, UMMA M=64 N=192 K=16, B = V as stored (keys x dims): MN-major descriptor
//   out = O / (rowsum * 64 * 1024)  -> fp32 and / or fp16 planes for the out-projection GEMM
// Accuracy is that of the GEMM engine (2^-22 relative per product), so the fp32 parity gates hold.
//
// One CTA per (clip, head), 160 threads: warps 0-3 = softmax / epilogue (TMEM lane quarter = warp, 16 rows each:
// a 64-row accumulator occupies lanes 0-15 of every quarter), warp 4 = TMA producer + MMA issuer.
#include "pm_common.cuh"
#include "pm_tc_ptx.cuh"
#include "../../include/pm_emage.h"

namespace {

constexpr int T = 64;                   // tokens per tile (queries and keys)
constexpr int HD = 192;                 // head dim
constexpr int KB = HD / 64;             // 64-column blocks per head
constexpr int BLK = T * 128;            // bytes of one 64 x 64 fp16 block (128-byte rows, 128B swizzle): 8 KB
constexpr int NTHREADS = 160;
constexpr float P_SCALE = 1024.f;       // probabilities are split as fp16 planes of 1024 * p (second plane stays normal)

struct Smem {
  static constexpr int Q = 0;                          // [2 planes][KB blocks]
  static constexpr int K = Q + 2 * KB * BLK;
  static constexpr int V = K + 2 * KB * BLK;
  static constexpr int P = V + 2 * KB * BLK;           // [2 planes] one block each
  static constexpr int BARS = P + 2 * BLK;             // qk_full[KB], v_full, s_full, p_full, o_full
  static constexpr int MISC = BARS + (KB + 4) * 8;
  static constexpr int TOTAL = MISC + 16;
};

// Instrumented build only (-DPM_ATTN_TIMING, tools/bench_attention.py --timeline): clock64 stamps of CTA 0's phases.
#ifdef PM_ATTN_TIMING
__device__ unsigned long long pm_attn_stamps[16];
#define AT_STAMP(i) do { if (blockIdx.x == 0 && (threadIdx.x & 31) == 0) pm_attn_stamps[i] = (unsigned long long)clock64(); } while (0)
#else
#define AT_STAMP(i) do {} while (0)
#endif

struct AttnParams {
  int heads, tq, tk;
  int qc0, kc0, vc0;                    // first column of head 0 inside the Q / K / V plane tensors
  float scale;                          // 1 / (sqrt(hd) * 64 * 64): the operand planes hold 64 x
  float* out; int ldo;                  // fp32 (batch*tq, >= heads*hd) or null
  PmPlanes planes;                      // fp16 planes of the output or ptr == null
  const int* q_len; const int* k_len;   // ragged batches (pm_attention_tc_rl, nullable): per-clip query / key counts
};

__device__ __forceinline__ void tmem_ld64(uint32_t taddr, uint32_t (&r)[64]) {
  uint32_t(&a)[32] = *reinterpret_cast<uint32_t(*)[32]>(&r[0]);
  uint32_t(&b)[32] = *reinterpret_cast<uint32_t(*)[32]>(&r[32]);
  tmem_ld32(taddr, a);
  tmem_ld32(taddr + 32, b);
}
__device__ __forceinline__ void sts128u(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

__global__ void __launch_bounds__(NTHREADS, 1) attention_tc_kernel(const __grid_constant__ CUtensorMap map_q,
                                                                   const __grid_constant__ CUtensorMap map_k,
                                                                   const __grid_constant__ CUtensorMap map_v,
                                                                   const AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t sm_u = smem_u32(sm);
  const uint32_t bars = sm_u + Smem::BARS;
  const uint32_t qk_full = bars, v_full = bars + 8 * KB, s_full = v_full + 8, p_full = v_full + 16, o_full = v_full + 24;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + Smem::MISC);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x / p.heads, h = blockIdx.x % p.heads;
  if (warp == 0) AT_STAMP(0);                              // kernel entry

  if (threadIdx.x == 0) {
    for (int kb = 0; kb < KB; ++kb) mbar_init(qk_full + 8 * kb, 1);
    mbar_init(v_full, 1);
    mbar_init(s_full, 1);
    mbar_init(p_full, 4);
    mbar_init(o_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(256) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_s = tmem_base, tmem_o = tmem_base + 64;
  if (warp == 0) AT_STAMP(1);                              // prologue done

  if (warp == 4) {
    // ===== TMA producer + MMA issuer =====
    if (elect_one()) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&map_q) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&map_k) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&map_v) : "memory");
      for (int kb = 0; kb < KB; ++kb) {                   // one barrier per 64-column block: the first MMAs start on a third of Q, K
        mbar_expect_tx(qk_full + 8 * kb, 4 * BLK);
        for (int pl = 0; pl < 2; ++pl) {
          tma_load_4d(sm_u + Smem::Q + (pl * KB + kb) * BLK, &map_q, qk_full + 8 * kb, p.qc0 + h * HD + kb * 64, 0, b, pl);
          tma_load_4d(sm_u + Smem::K + (pl * KB + kb) * BLK, &map_k, qk_full + 8 * kb, p.kc0 + h * HD + kb * 64, 0, b, pl);
        }
      }
      mbar_expect_tx(v_full, 2 * KB * BLK);
      for (int pl = 0; pl < 2; ++pl)
        for (int nb = 0; nb < KB; ++nb)
          tma_load_4d(sm_u + Smem::V + (pl * KB + nb) * BLK, &map_v, v_full, p.vc0 + h * HD + nb * 64, 0, b, pl);
    }
    __syncwarp();
    // ---- S = Q K^T : D = f32, A = B = f16, both K-major, N = 64, M = 64
    {
      constexpr uint32_t IDESC_S = (1u << 4) | ((uint32_t)(T >> 3) << 17) | ((uint32_t)(T >> 4) << 24);
      const uint64_t q0 = UMMA_DESC_K_SW128 | (uint64_t)(((sm_u + Smem::Q) >> 4) & 0x3FFFu);
      const uint64_t k0 = UMMA_DESC_K_SW128 | (uint64_t)(((sm_u + Smem::K) >> 4) & 0x3FFFu);
      constexpr uint64_t PL = (uint64_t)(KB * BLK) >> 4, KBS = (uint64_t)BLK >> 4;
      // per block: cross products first (small), the main product last: (A plane, B plane) = (0,1), (1,0), (0,0)
      const int pa[3] = {0, 1, 0}, pb[3] = {1, 0, 0};
      uint32_t acc = 0;
#pragma unroll
      for (int kb = 0; kb < KB; ++kb) {
        mbar_wait(qk_full + 8 * kb, 0);
        tc_fence_after();
        AT_STAMP(8 + kb);                                  // Q | K block kb landed
        if (elect_one()) {
#pragma unroll
          for (int t = 0; t < 3; ++t)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              tc_mma_bf16(tmem_s, q0 + pa[t] * PL + kb * KBS + k * 2, k0 + pb[t] * PL + kb * KBS + k * 2, IDESC_S, acc);
              acc = 1;
            }
          if (kb == KB - 1) tc_commit(s_full);
        }
        __syncwarp();
      }
    }
    // ---- O = P V : B = V as stored, (keys x dims) = MN-major: 64-dim groups 8 KB apart (LBO), 8-key groups 1 KB (SBO)
    mbar_wait(v_full, 0);
    mbar_wait(p_full, 0);
    tc_fence_after();
    if (elect_one()) {
      constexpr uint32_t IDESC_O = (1u << 4) | (1u << 16) | ((uint32_t)(HD >> 3) << 17) | ((uint32_t)(T >> 4) << 24);
      constexpr uint64_t DESC_MN = ((uint64_t)(BLK >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
      const uint64_t p0 = UMMA_DESC_K_SW128 | (uint64_t)(((sm_u + Smem::P) >> 4) & 0x3FFFu);
      const uint64_t v0 = DESC_MN | (uint64_t)(((sm_u + Smem::V) >> 4) & 0x3FFFu);
      constexpr uint64_t PPL = (uint64_t)BLK >> 4, VPL = (uint64_t)(KB * BLK) >> 4;
      const int pa[3] = {0, 1, 0}, pb[3] = {1, 0, 0};
      uint32_t acc = 0;
#pragma unroll
      for (int t = 0; t < 3; ++t)
#pragma unroll
        for (int k = 0; k < 4; ++k) {       // 16 keys per step: A advances 32 B inside the swizzled row, B by two 8-key groups
          tc_mma_bf16(tmem_o, p0 + pa[t] * PPL + k * 2, v0 + pb[t] * VPL + k * (2048 >> 4), IDESC_O, acc);
          acc = 1;
        }
      tc_commit(o_full);
    }
    __syncwarp();
  } else {
    // ===== softmax + epilogue: warp w owns query rows 16 w .. 16 w + 15 (TMEM lanes 32 w + 0..15) =====
    const int row = warp * 16 + (lane & 15);
    const bool active = lane < 16;
    const uint32_t lane_addr = (uint32_t)(warp * 32) << 16;
    float inv = 0.f;
    {
      mbar_wait(s_full, 0);
      tc_fence_after();
      if (warp == 0) AT_STAMP(2);                          // S complete
      uint32_t sr[64];
      tmem_ld64(tmem_s + lane_addr, sr);
      // exp(s - m) = 2^((s - m) log2 e): log2 e is folded into the scale and the exponential is one MUFU.EX2
      // (2 ulp); expf() costs ~25 instructions per element on 16 active lanes - the softmax was 5 400 of the kernel's
      // 20 000 cycles (profiles/r2/attention_timeline.md)
      const float sl2 = p.scale * 1.4426950408889634f;
      const int tk = p.k_len ? min(p.tk, __ldg(p.k_len + b)) : p.tk;      // keys beyond a clip's count: probability 0
      float m = -INFINITY;
#pragma unroll
      for (int j = 0; j < 64; ++j) {
        const float v = j < tk ? __uint_as_float(sr[j]) * sl2 : -INFINITY;
        sr[j] = __float_as_uint(v);
        m = fmaxf(m, v);
      }
      float sum = 0.f;
#pragma unroll
      for (int j = 0; j < 64; ++j) {
        float e = 0.f;
        if (j < tk) asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(__uint_as_float(sr[j]) - m));
        sum += e;
        sr[j] = __float_as_uint(e * P_SCALE);
      }
      inv = tk > 0 ? 1.f / (sum * (P_SCALE * PM_F16_ACT_SCALE)) : 0.f;
      if (active) {
        const uint32_t dst = sm_u + Smem::P + (row >> 3) * 1024 + (row & 7) * 128;
#pragma unroll
        for (int c = 0; c < 8; ++c) {       // 8 keys per 16-byte chunk, two planes
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const float a0 = __uint_as_float(sr[8 * c + 2 * u]), a1 = __uint_as_float(sr[8 * c + 2 * u + 1]);
            const float f0 = pm_f16_head(a0), f1 = pm_f16_head(a1);       // exact in fp16: no conversion back (pm_common.cuh)
            const __half2 h0 = __floats2half2_rn(f0, f1);
            const __half2 h1 = __floats2half2_rn(a0 - f0, a1 - f1);
            hi[u] = *reinterpret_cast<const uint32_t*>(&h0);
            lo[u] = *reinterpret_cast<const uint32_t*>(&h1);
          }
          const uint32_t off = (uint32_t)((c ^ (row & 7)) << 4);
          sts128u(dst + off, hi[0], hi[1], hi[2], hi[3]);
          sts128u(dst + BLK + off, lo[0], lo[1], lo[2], lo[3]);
        }
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
      if (warp == 0) AT_STAMP(3);                          // softmax done, P stored
    }
    // ---- O: normalise and write straight from registers (thread = query row): 16-byte vectors per plane / float4 for
    // fp32.  (Staging the tile in shared memory and copying it out row-contiguously cost 9 600 of 20 000 cycles.)
    mbar_wait(o_full, 0);
    tc_fence_after();
    if (warp == 0) AT_STAMP(4);                            // O complete
    const bool live = active && row < p.tq;
    // ragged batches: query rows beyond the clip's count (and every row of a clip without keys) are written as 0
    const bool zero = (p.q_len && row >= __ldg(p.q_len + b)) || (p.k_len && __ldg(p.k_len + b) <= 0);
    const long long grow = (long long)b * p.tq + row;
    const bool vec16 = p.planes.ptr && ((p.planes.ld & 7) == 0) && ((p.planes.ps & 7) == 0) &&
                       ((reinterpret_cast<uintptr_t>(p.planes.ptr) & 15) == 0);
    __half* const prow = reinterpret_cast<__half*>(p.planes.ptr) + grow * p.planes.ld + h * HD;
    float* const frow = p.out ? p.out + grow * p.ldo + h * HD : nullptr;
#pragma unroll 1
    for (int c0 = 0; c0 < HD; c0 += 64) {
      uint32_t orr[64];
      tmem_ld64(tmem_o + lane_addr + c0, orr);
      if (live) {
#pragma unroll
        for (int g8 = 0; g8 < 8; ++g8) {                   // 8 consecutive columns
          float x[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) x[u] = zero ? 0.f : __uint_as_float(orr[8 * g8 + u]) * inv;
          if (frow) {
            *reinterpret_cast<float4*>(frow + c0 + 8 * g8) = make_float4(x[0], x[1], x[2], x[3]);
            *reinterpret_cast<float4*>(frow + c0 + 8 * g8 + 4) = make_float4(x[4], x[5], x[6], x[7]);
          }
          if (p.planes.ptr) {
            if (vec16) {
              uint32_t h0[4], h1[4];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const float a0 = x[2 * u] * PM_F16_ACT_SCALE, a1 = x[2 * u + 1] * PM_F16_ACT_SCALE;
                const float f0 = pm_f16_head(a0), f1 = pm_f16_head(a1);
                const __half2 t0 = __floats2half2_rn(f0, f1);
                const __half2 t1 = __floats2half2_rn(a0 - f0, a1 - f1);
                h0[u] = *reinterpret_cast<const uint32_t*>(&t0);
                h1[u] = *reinterpret_cast<const uint32_t*>(&t1);
              }
              *reinterpret_cast<uint4*>(prow + c0 + 8 * g8) = make_uint4(h0[0], h0[1], h0[2], h0[3]);
              if (p.planes.nsplit > 1) *reinterpret_cast<uint4*>(prow + p.planes.ps + c0 + 8 * g8) = make_uint4(h1[0], h1[1], h1[2], h1[3]);
            } else {
#pragma unroll
              for (int u = 0; u < 8; ++u) pm_store_planes_t<true>(p.planes, grow, h * HD + c0 + 8 * g8 + u, x[u]);
            }
          }
        }
      }
    }
    if (warp == 0) AT_STAMP(5);
  }

  if (warp == 0) AT_STAMP(6);                              // outputs written
  tc_fence_before();
  __syncthreads();
  if (warp == 0) AT_STAMP(7);
  if (warp == 4) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(256) : "memory");
  }
}

constexpr size_t kSmem = Smem::TOTAL + 1024;

// (cols, rows of one clip, clips, planes) view of a two-plane fp16 activation; box = 64 cols x 64 rows of one clip
bool plane_map(CUtensorMap* m, const uint16_t* base, long long ps, long long bs, int ld, int cols, int rows, int batch) {
  cuuint64_t dims[4] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batch, 2};
  cuuint64_t strides[3] = {(cuuint64_t)ld * 2, (cuuint64_t)bs * 2, (cuuint64_t)ps * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)T, 1, 1};
  return encode_map(m, base, 4, dims, strides, box, true);
}

}  // namespace

static int attention_tc_run(const uint16_t* Q, long long q_ps, long long q_bs, int ldq, int q_cols, int q_col0,
                            const uint16_t* K, long long k_ps, long long k_bs, int ldk, int k_cols, int k_col0,
                            const uint16_t* V, long long v_ps, long long v_bs, int ldv, int v_cols, int v_col0,
                            float* O, int ldo, int batch, int heads, int tq, int tk, int head_dim,
                            uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, const int* q_len, const int* k_len,
                            void* stream) {
  PM_REQUIRE(Q && K && V && (O || planes) && batch >= 0 && heads > 0);
  PM_TAKE_FMT(p_nsplit, f16);
  PM_REQUIRE(!planes || (f16 && p_nsplit <= 2));           // fp16 planes in, (at most two) fp16 planes out
  PM_REQUIRE(pm_planes_ok(planes, p_ps, p_ld, p_nsplit, heads * head_dim, false));
  if (head_dim != HD || tq > T || tk > T || tq <= 0 || tk <= 0) return PM_EUNSUPPORTED;
  PM_REQUIRE(!O || (ldo & 3) == 0);
  // TMA: 16-byte aligned bases and strides; the head slices must lie inside the tensors
  for (const void* ptr : {(const void*)Q, (const void*)K, (const void*)V}) PM_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0);
  PM_REQUIRE((ldq & 7) == 0 && (ldk & 7) == 0 && (ldv & 7) == 0 && (q_ps & 7) == 0 && (k_ps & 7) == 0 && (v_ps & 7) == 0);
  PM_REQUIRE(batch <= 1 || ((q_bs & 7) == 0 && (k_bs & 7) == 0 && (v_bs & 7) == 0));
  PM_REQUIRE(q_col0 >= 0 && k_col0 >= 0 && v_col0 >= 0 && q_col0 + heads * HD <= q_cols && k_col0 + heads * HD <= k_cols &&
             v_col0 + heads * HD <= v_cols && q_cols <= ldq && k_cols <= ldk && v_cols <= ldv);
  if (batch == 0) return PM_OK;
  CUtensorMap mq, mk, mv;
  if (!plane_map(&mq, Q, q_ps, q_bs, ldq, q_cols, tq, batch) || !plane_map(&mk, K, k_ps, k_bs, ldk, k_cols, tk, batch) ||
      !plane_map(&mv, V, v_ps, v_bs, ldv, v_cols, tk, batch))
    return PM_EBADARG;
  AttnParams p;
  p.heads = heads; p.tq = tq; p.tk = tk; p.qc0 = q_col0; p.kc0 = k_col0; p.vc0 = v_col0;
  p.scale = 1.0f / (sqrtf((float)head_dim) * PM_F16_ACT_SCALE * PM_F16_ACT_SCALE);
  p.out = O; p.ldo = ldo;
  p.planes = PmPlanes{reinterpret_cast<__nv_bfloat16*>(planes), p_ps, p_ld, p_nsplit};
  p.q_len = q_len; p.k_len = k_len;
  static unsigned long long configured = 0;
  if (pm_first_use_on_device(configured)) {
    cudaError_t e = cudaFuncSetAttribute(attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem);
    if (e != cudaSuccess) { configured = 0; return (int)e; }
  }
  attention_tc_kernel<<<batch * heads, NTHREADS, kSmem, (cudaStream_t)stream>>>(mq, mk, mv, p);
  PM_LAUNCH_CHECK();
}

extern "C" int pm_attention_tc(const uint16_t* Q, long long q_ps, long long q_bs, int ldq, int q_cols, int q_col0,
                               const uint16_t* K, long long k_ps, long long k_bs, int ldk, int k_cols, int k_col0,
                               const uint16_t* V, long long v_ps, long long v_bs, int ldv, int v_cols, int v_col0,
                               float* O, int ldo, int batch, int heads, int tq, int tk, int head_dim,
                               uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream) {
  return attention_tc_run(Q, q_ps, q_bs, ldq, q_cols, q_col0, K, k_ps, k_bs, ldk, k_cols, k_col0, V, v_ps, v_bs, ldv,
                          v_cols, v_col0, O, ldo, batch, heads, tq, tk, head_dim, planes, p_ps, p_ld, p_nsplit, nullptr,
                          nullptr, stream);
}

extern "C" int pm_attention_tc_rl(const uint16_t* Q, long long q_ps, long long q_bs, int ldq, int q_cols, int q_col0,
                                  const uint16_t* K, long long k_ps, long long k_bs, int ldk, int k_cols, int k_col0,
                                  const uint16_t* V, long long v_ps, long long v_bs, int ldv, int v_cols, int v_col0,
                                  float* O, int ldo, int batch, int heads, int tq, int tk, int head_dim,
                                  uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, const int* q_len,
                                  const int* k_len, void* stream) {
  return attention_tc_run(Q, q_ps, q_bs, ldq, q_cols, q_col0, K, k_ps, k_bs, ldk, k_cols, k_col0, V, v_ps, v_bs, ldv,
                          v_cols, v_col0, O, ldo, batch, heads, tq, tk, head_dim, planes, p_ps, p_ld, p_nsplit, q_len,
                          k_len, stream);
}

#ifdef PM_ATTN_TIMING
extern "C" int pm_attn_timing_read(unsigned long long* host) {
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return (int)e;
  return (int)cudaMemcpyFromSymbol(host, pm_attn_stamps, sizeof(unsigned long long) * 16);
}
#endif
