// Whole-sequence multi-head attention for the EMAGE transformer layers: fp32 SIMT kernel of the fp32 / bf16-plane
// engines (the default fp16x3 engine runs attention on the tensor cores, pm_attention_tc.cu; an mma.sync 3xTF32
// variant of this kernel measured 1.3 % faster per step in round 2 and was removed in favour of the tcgen05 kernel).
// T <= 64 tokens, head_dim = 192, no masks: the full score tile lives on chip, so there is no
// online-softmax pass.  One CTA per (clip, head).  Contract: include/pm_emage.h (pm_attention_f32).
#include <stdlib.h>
#include "pm_common.cuh"
#include "../../include/pm_emage.h"

namespace {

constexpr int TMAX = 64;
constexpr int HD = 192;
constexpr int HDP = HD + 1;     // +1 float: conflict-free column walks over rows
constexpr int NT = 256;

template <bool F16>
__global__ void __launch_bounds__(NT) attention_f32_kernel(
    const float* __restrict__ Q, int ldq, const float* __restrict__ K, int ldk,
    const float* __restrict__ V, int ldv, float* __restrict__ O, int ldo,
    int heads, int tq, int tk, float scale, PmPlanes P, const int* __restrict__ q_len, const int* __restrict__ k_len) {
  extern __shared__ float smem[];
  float* Qs = smem;                    // [TMAX][HDP]
  float* Ks = Qs + TMAX * HDP;         // [TMAX][HDP]
  float* Vs = Ks + TMAX * HDP;         // [TMAX][HD]
  float* S = Vs + TMAX * HD;           // [TMAX][TMAX+1]
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  const int tid = threadIdx.x;
  // ragged batches (pm_attention_f32_rl): keys beyond the clip's count get probability 0, query rows beyond its count
  // (every row when it has no key) are written as 0
  const int tkv = k_len ? min(tk, __ldg(k_len + b)) : tk;
  const int tqv = q_len ? min(tq, __ldg(q_len + b)) : tq;

  // stage Q, K, V head slices (float4 global loads, scalar smem stores because of the +1 padding)
  for (int i = tid; i < TMAX * (HD / 4); i += NT) {
    const int r = i / (HD / 4), c4 = i % (HD / 4);
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f), k = q, v = q;
    if (r < tq) q = *reinterpret_cast<const float4*>(Q + (long long)(b * tq + r) * ldq + h * HD + c4 * 4);
    if (r < tk) {
      k = *reinterpret_cast<const float4*>(K + (long long)(b * tk + r) * ldk + h * HD + c4 * 4);
      v = *reinterpret_cast<const float4*>(V + (long long)(b * tk + r) * ldv + h * HD + c4 * 4);
    }
    float* qd = Qs + r * HDP + c4 * 4;
    qd[0] = q.x; qd[1] = q.y; qd[2] = q.z; qd[3] = q.w;
    float* kd = Ks + r * HDP + c4 * 4;
    kd[0] = k.x; kd[1] = k.y; kd[2] = k.z; kd[3] = k.w;
    *reinterpret_cast<float4*>(Vs + r * HD + c4 * 4) = v;
  }
  __syncthreads();

  // S = scale * Q K^T : each thread a 4x4 block of the 64x64 tile
  {
    const int ti = tid >> 4, tj = tid & 15;
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[a][c] = 0.f;
    const float* q0 = Qs + (ti * 4) * HDP;
    const float* k0 = Ks + (tj * 4) * HDP;
#pragma unroll 4
    for (int d = 0; d < HD; ++d) {
      float qv[4], kv[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) { qv[a] = q0[a * HDP + d]; kv[a] = k0[a * HDP + d]; }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][c] = fmaf(qv[a], kv[c], acc[a][c]);
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c) S[(ti * 4 + a) * (TMAX + 1) + tj * 4 + c] = acc[a][c] * scale;
  }
  __syncthreads();

  // row softmax over the tk valid keys: warp w owns rows w, w+8, ...
  {
    const int warp = tid >> 5, lane = tid & 31;
    for (int r = warp; r < tq; r += NT / 32) {
      float* row = S + r * (TMAX + 1);
      const float v0 = lane < tkv ? row[lane] : -INFINITY;
      const float v1 = lane + 32 < tkv ? row[lane + 32] : -INFINITY;
      const float m = pm_warp_max(fmaxf(v0, v1));
      const float e0 = lane < tkv ? expf(v0 - m) : 0.f;
      const float e1 = lane + 32 < tkv ? expf(v1 - m) : 0.f;
      const float inv = 1.f / pm_warp_sum(e0 + e1);
      row[lane] = e0 * inv;
      row[lane + 32] = e1 * inv;
    }
  }
  __syncthreads();

  // O = P V : thread -> 4 rows x 12 strided columns
  {
    const int tr = tid >> 4, tc = tid & 15;
    float acc[4][12];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int m = 0; m < 12; ++m) acc[a][m] = 0.f;
    for (int j = 0; j < tkv; ++j) {
      float pv[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) pv[a] = S[(tr * 4 + a) * (TMAX + 1) + j];
#pragma unroll
      for (int m = 0; m < 12; ++m) {
        const float vv = Vs[j * HD + tc + 16 * m];
#pragma unroll
        for (int a = 0; a < 4; ++a) acc[a][m] = fmaf(pv[a], vv, acc[a][m]);
      }
    }
    // stage the 64 x 192 output tile in smem (the Q region is dead by now) so global writes are row-contiguous
    __syncthreads();
    float* Os = Qs;                      // [TMAX][HD]
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int m = 0; m < 12; ++m) Os[(tr * 4 + a) * HD + tc + 16 * m] = acc[a][m];
  }
  __syncthreads();
  {
    const float* Os = Qs;
    const bool vec_p = P.ptr && ((P.ld & 3) == 0) && ((P.ps & 3) == 0) && ((reinterpret_cast<uintptr_t>(P.ptr) & 7) == 0);
    for (int i = tid; i < tq * (HD / 4); i += NT) {
      const int r = i / (HD / 4), c4 = i % (HD / 4);
      const float4 v = (r < tqv && tkv > 0) ? *reinterpret_cast<const float4*>(Os + r * HD + c4 * 4)
                                             : make_float4(0.f, 0.f, 0.f, 0.f);
      const long long row = (long long)b * tq + r;
      if (O) *reinterpret_cast<float4*>(O + row * ldo + h * HD + c4 * 4) = v;
      if (P.ptr) {
        if (vec_p) pm_store_planes4_t<F16>(P, row, h * HD + c4 * 4, v);
        else {
          pm_store_planes_t<F16>(P, row, h * HD + c4 * 4, v.x); pm_store_planes_t<F16>(P, row, h * HD + c4 * 4 + 1, v.y);
          pm_store_planes_t<F16>(P, row, h * HD + c4 * 4 + 2, v.z); pm_store_planes_t<F16>(P, row, h * HD + c4 * 4 + 3, v.w);
        }
      }
    }
  }
}

constexpr size_t kSmemBytes = (size_t)(2 * TMAX * HDP + TMAX * HD + TMAX * (TMAX + 1)) * sizeof(float);

}  // namespace

static int attention_f32_run(const float* Q, int ldq, const float* K, int ldk, const float* V, int ldv,
                             float* O, int ldo, int batch, int heads, int tq, int tk, int head_dim,
                             uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, const int* q_len, const int* k_len,
                             void* stream) {
  PM_REQUIRE(Q && K && V && (O || planes) && batch >= 0 && heads > 0);
  PM_TAKE_FMT(p_nsplit, f16);
  PM_REQUIRE(pm_planes_ok(planes, p_ps, p_ld, p_nsplit, heads * head_dim, false));
  const PmPlanes P{reinterpret_cast<__nv_bfloat16*>(planes), p_ps, p_ld, p_nsplit};
  if (head_dim != HD || tq > TMAX || tk > TMAX || tq <= 0 || tk <= 0) return PM_EUNSUPPORTED;
  PM_REQUIRE((ldq & 3) == 0 && (ldk & 3) == 0 && (ldv & 3) == 0 && (!O || (ldo & 3) == 0));
  if (batch == 0) return PM_OK;
  static unsigned long long configured = 0;
  if (pm_first_use_on_device(configured)) {
    cudaError_t e = cudaFuncSetAttribute(attention_f32_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)kSmemBytes);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attention_f32_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes);
    if (e != cudaSuccess) { configured = 0; return (int)e; }
  }
  if (f16) attention_f32_kernel<true><<<batch * heads, NT, kSmemBytes, (cudaStream_t)stream>>>(
      Q, ldq, K, ldk, V, ldv, O, ldo, heads, tq, tk, 1.0f / sqrtf((float)head_dim), P, q_len, k_len);
  else attention_f32_kernel<false><<<batch * heads, NT, kSmemBytes, (cudaStream_t)stream>>>(
      Q, ldq, K, ldk, V, ldv, O, ldo, heads, tq, tk, 1.0f / sqrtf((float)head_dim), P, q_len, k_len);
  PM_LAUNCH_CHECK();
}

extern "C" int pm_attention_f32(const float* Q, int ldq, const float* K, int ldk, const float* V, int ldv,
                                float* O, int ldo, int batch, int heads, int tq, int tk, int head_dim,
                                uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream) {
  return attention_f32_run(Q, ldq, K, ldk, V, ldv, O, ldo, batch, heads, tq, tk, head_dim, planes, p_ps, p_ld, p_nsplit,
                           nullptr, nullptr, stream);
}

extern "C" int pm_attention_f32_rl(const float* Q, int ldq, const float* K, int ldk, const float* V, int ldv,
                                   float* O, int ldo, int batch, int heads, int tq, int tk, int head_dim,
                                   uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, const int* q_len,
                                   const int* k_len, void* stream) {
  return attention_f32_run(Q, ldq, K, ldk, V, ldv, O, ldo, batch, heads, tq, tk, head_dim, planes, p_ps, p_ld, p_nsplit,
                           q_len, k_len, stream);
}
