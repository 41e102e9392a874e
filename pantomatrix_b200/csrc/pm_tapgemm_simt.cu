// fp32 SIMT tap-GEMM: the exact-order reference engine for Conv1d / Linear on the EMAGE path.
// See include/pm_emage.h (pm_tapgemm_f32) for the contract and the reference call sites.
//
// Tiling: CTA = 128 output rows x 64 output channels, K step 16 over (tap, cin) pairs; 256 threads,
// 8x4 register micro-tile per thread.  Grid = (row tiles, channel tiles, batch).
#include "pm_common.cuh"
#include "../../include/pm_emage.h"

namespace {

constexpr int BM = 128, BN = 64, BK = 16, NT = 256;

struct TapGemmParams {
  const float* A; long long a_bs; int lda; int rows_in; int cin;
  const float* W; const float* bias; int taps; int stride; int pad;
  int rows_out; int cout;
  const float* R; long long r_bs; int ldr;
  int act; float slope;
  float* O; long long o_bs; int ldo;
  const int* row_limit; int rows_per_clip;   // ragged batches (pm_tapgemm_f32_rl), see pm_tapgemm_tc.cu
};

__global__ void __launch_bounds__(NT) tapgemm_f32_kernel(TapGemmParams p) {
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Ws[BK][BN + 4];

  const int tid = threadIdx.x;
  const int l0 = blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;
  const int b = blockIdx.z;
  const float* __restrict__ A = p.A + (long long)b * p.a_bs;
  const int ty = tid >> 4;   // 16 row groups of 8
  const int tx = tid & 15;   // 16 col groups of 4

  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int kc = tid & 15;        // channel within the K tile
  const int kr = tid >> 4;        // 0..15

  for (int t = 0; t < p.taps; ++t) {
    const float* __restrict__ Wt = p.W + (long long)t * p.cout * p.cin;
    for (int c0 = 0; c0 < p.cin; c0 += BK) {
      const int c = c0 + kc;
      const bool c_ok = c < p.cin;
      // A tile: 128 rows x 16 channels, 8 loads per thread (consecutive threads -> consecutive channels)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = kr + i * 16;
        const int l = l0 + r;
        const int row = l * p.stride + t - p.pad;
        float v = 0.f;
        if (c_ok && l < p.rows_out && row >= 0 && row < p.rows_in) v = __ldg(A + (long long)row * p.lda + c);
        As[kc][r] = v;
      }
      // W tile: 64 out channels x 16 in channels
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int n = kr + i * 16;
        float v = 0.f;
        if (c_ok && n0 + n < p.cout) v = __ldg(Wt + (long long)(n0 + n) * p.cin + c);
        Ws[kc][n] = v;
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < BK; ++k) {
        const float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 8]);
        const float4 a1 = *reinterpret_cast<const float4*>(&As[k][ty * 8 + 4]);
        const float4 w = *reinterpret_cast<const float4*>(&Ws[k][tx * 4]);
        const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
      }
      __syncthreads();
    }
  }

  float* __restrict__ O = p.O + (long long)b * p.o_bs;
  const float* __restrict__ R = p.R ? p.R + (long long)b * p.r_bs : nullptr;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int l = l0 + ty * 8 + i;
    if (l >= p.rows_out) continue;
    bool zero = false;                     // beyond its clip's row limit: stored as 0 (negative limit: not stored)
    if (p.row_limit) {
      long long clip = b, r = l;
      if (p.rows_per_clip > 0) {
        const long long g = (long long)b * p.rows_out + l;
        clip = g / p.rows_per_clip;
        r = g - clip * p.rows_per_clip;
      }
      const int lim = __ldg(p.row_limit + clip);
      if (r >= lim) {
        if (lim < 0) continue;
        zero = true;
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= p.cout) continue;
      if (zero) { O[(long long)l * p.ldo + n] = 0.f; continue; }
      float v = acc[i][j];
      if (p.bias) v += __ldg(p.bias + n);
      if (R) v += __ldg(R + (long long)l * p.ldr + n);
      O[(long long)l * p.ldo + n] = pm_act(v, p.act, p.slope);
    }
  }
}

static int tapgemm_f32_run(const float* A, long long a_bs, int lda, int batch, int rows_in, int cin,
                           const float* W, const float* bias, int taps, int stride, int pad,
                           int rows_out, int cout,
                           const float* residual, long long r_bs, int ldr,
                           int act, float slope,
                           float* out, long long o_bs, int ldo, const int* row_limit, int rows_per_clip, void* stream) {
  PM_REQUIRE(rows_per_clip >= 0);
  PM_REQUIRE(A && W && out);
  PM_REQUIRE(batch >= 0 && rows_in >= 0 && rows_out >= 0 && cin > 0 && cout > 0 && taps > 0 && stride > 0);
  PM_REQUIRE(lda >= cin && ldo >= cout && (!residual || ldr >= cout));
  PM_REQUIRE(act >= PM_ACT_NONE && act <= PM_ACT_LEAKY);
  if (batch == 0 || rows_out == 0) return PM_OK;
  PM_REQUIRE(batch <= 65535);
  TapGemmParams p{A, a_bs, lda, rows_in, cin, W, bias, taps, stride, pad, rows_out, cout,
                  residual, r_bs, ldr, act, slope, out, o_bs, ldo, row_limit, rows_per_clip};
  dim3 grid(pm_cdiv(rows_out, BM), pm_cdiv(cout, BN), batch);
  tapgemm_f32_kernel<<<grid, NT, 0, (cudaStream_t)stream>>>(p);
  PM_LAUNCH_CHECK();
}

}  // namespace

extern "C" int pm_tapgemm_f32(const float* A, long long a_bs, int lda, int batch, int rows_in, int cin,
                              const float* W, const float* bias, int taps, int stride, int pad,
                              int rows_out, int cout,
                              const float* residual, long long r_bs, int ldr,
                              int act, float slope,
                              float* out, long long o_bs, int ldo, void* stream) {
  return tapgemm_f32_run(A, a_bs, lda, batch, rows_in, cin, W, bias, taps, stride, pad, rows_out, cout, residual, r_bs,
                         ldr, act, slope, out, o_bs, ldo, nullptr, 0, stream);
}

extern "C" int pm_tapgemm_f32_rl(const float* A, long long a_bs, int lda, int batch, int rows_in, int cin,
                                 const float* W, const float* bias, int taps, int stride, int pad,
                                 int rows_out, int cout,
                                 const float* residual, long long r_bs, int ldr,
                                 int act, float slope,
                                 float* out, long long o_bs, int ldo, const int* row_limit, int rows_per_clip,
                                 void* stream) {
  return tapgemm_f32_run(A, a_bs, lda, batch, rows_in, cin, W, bias, taps, stride, pad, rows_out, cout, residual, r_bs,
                         ldr, act, slope, out, o_bs, ldo, row_limit, rows_per_clip, stream);
}
