// Small HBM-bound kernels of the EMAGE path: WavEncoder stem, residual LayerNorm, broadcast adds,
// window assembly.  Contracts and reference call sites: include/pm_emage.h.
#include "pm_common.cuh"
#include "../../include/pm_emage.h"

namespace {

// ---------------------------------------------------------------------------------------------------
// WavEncoder stem (Cin = 1): both convs of the first block share the input samples.
//
// Round 1 ran one thread per (row, channel) with weights and samples in shared memory: 45 shared loads for 30 FMAs per
// output, 370 us for the 0.97 M rows x 64 channels of the BASELINE batch against ~80 us of output traffic (sc fp32 +
// operand planes), plus a separate 97 us fp32 -> planes pass.  Now: a lane owns a channel PAIR with the 60 weights in
// registers, a warp walks the tile three rows at a time (25 broadcast sample loads for 180 FMAs) and the conv1 output
// goes out as the next GEMM's operand planes directly.  The fmaf order per output (k = 0 .. 14, then the bias) is the
// old kernel's, so results are unchanged bit for bit.
// ---------------------------------------------------------------------------------------------------
constexpr int STEM_ROWS = 192;            // rows per CTA
constexpr int STEM_THREADS = 256;

template <bool F16>
__device__ __forceinline__ void stem_store_planes2(const PmPlanes& P, long long row, int c, float a, float b) {
  if constexpr (F16) {
    if (P.nsplit == 2) {                  // two fp16 planes: 4-byte stores, plane 0 by bit mask (pm_f16_head)
      __half* o = reinterpret_cast<__half*>(P.ptr) + row * P.ld + c;
      a *= PM_F16_ACT_SCALE; b *= PM_F16_ACT_SCALE;
      const float a0 = pm_f16_head(a), b0 = pm_f16_head(b);
      *reinterpret_cast<__half2*>(o) = __floats2half2_rn(a0, b0);
      *reinterpret_cast<__half2*>(o + P.ps) = __floats2half2_rn(a - a0, b - b0);
      return;
    }
  }
  pm_store_planes_t<F16>(P, row, c, a);
  pm_store_planes_t<F16>(P, row, c + 1, b);
}

template <int KS, int COUT, bool F16>
__global__ void __launch_bounds__(STEM_THREADS, 2) wav_stem_kernel(
    const float* __restrict__ audio, long long a_bs, long long a_ws, int batch, int n_samples,
    const float* __restrict__ w1, const float* __restrict__ b1, const float* __restrict__ wd,
    const float* __restrict__ bd, int stride, int pad, int rows_out, float slope,
    float* __restrict__ y1, float* __restrict__ sc, const PmPlanes P, const int* __restrict__ n_valid) {
  extern __shared__ float sx[];            // the input span of this tile: (STEM_ROWS - 1) * stride + KS samples
  constexpr int LPR = COUT / 2;            // lanes per row (a lane owns channels 2*cp, 2*cp + 1)
  constexpr int RW = 32 / LPR;             // row groups per warp
  constexpr int RPI = 3 * RW * (STEM_THREADS / 32);   // rows per CTA iteration
  static_assert(STEM_ROWS % RPI == 0, "tile must be whole iterations");
  const int seq = blockIdx.y;              // w*batch + b: window-major, so one window's clips are contiguous
  const int w = seq / batch, b = seq % batch;
  const float* __restrict__ x = audio + (long long)b * a_bs + (long long)w * a_ws;
  const int l0 = blockIdx.x * STEM_ROWS;
  const int span = (STEM_ROWS - 1) * stride + KS;
  // ragged batches: the slice holds n_valid[seq] samples (the rest reads as the reference's zero padding) and only
  // the rows the shorter slice yields are valid; the others are written as 0 for the convolutions that follow
  int n_in = n_samples, valid_rows = rows_out;
  if (n_valid) {
    n_in = min(n_samples, __ldg(n_valid + seq));
    const int num = n_in + 2 * pad - KS;
    valid_rows = n_in <= 0 || num < 0 ? 0 : min(rows_out, num / stride + 1);
  }
  for (int i = threadIdx.x; i < span; i += STEM_THREADS) {
    const int s = l0 * stride - pad + i;
    sx[i] = (s >= 0 && s < n_in) ? x[s] : 0.f;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cp = lane % LPR, rs = lane / LPR;
  const int c0 = 2 * cp;
  float wa0[KS], wa1[KS], wb0[KS], wb1[KS];   // conv1 / downsample weights of the two channels
#pragma unroll
  for (int k = 0; k < KS; ++k) {
    wa0[k] = __ldg(w1 + c0 * KS + k);
    wa1[k] = __ldg(w1 + (c0 + 1) * KS + k);
    wb0[k] = __ldg(wd + c0 * KS + k);
    wb1[k] = __ldg(wd + (c0 + 1) * KS + k);
  }
  const float ba0 = __ldg(b1 + c0), ba1 = __ldg(b1 + c0 + 1), bb0 = __ldg(bd + c0), bb1 = __ldg(bd + c0 + 1);
  __syncthreads();
#pragma unroll 1
  for (int it = 0; it < STEM_ROWS / RPI; ++it) {
    const int r0 = (it * (STEM_THREADS / 32) + warp) * 3 * RW + rs * 3;      // first of this lane's three rows (in tile)
    if (l0 + r0 >= rows_out) continue;
    const float* xr = sx + r0 * stride;
    float acc[3][4];
#pragma unroll
    for (int j = 0; j < 3; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
    if (stride == 5) {                     // the reference's stem: rows share samples, 25 loads for three rows
      float xv[2 * 5 + KS];
#pragma unroll
      for (int i = 0; i < 2 * 5 + KS; ++i) xv[i] = xr[i];
#pragma unroll
      for (int j = 0; j < 3; ++j) {
#pragma unroll
        for (int k = 0; k < KS; ++k) {
          const float v = xv[5 * j + k];
          acc[j][0] = fmaf(v, wa0[k], acc[j][0]);
          acc[j][1] = fmaf(v, wa1[k], acc[j][1]);
          acc[j][2] = fmaf(v, wb0[k], acc[j][2]);
          acc[j][3] = fmaf(v, wb1[k], acc[j][3]);
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 3; ++j) {
#pragma unroll
        for (int k = 0; k < KS; ++k) {
          const float v = xr[j * stride + k];
          acc[j][0] = fmaf(v, wa0[k], acc[j][0]);
          acc[j][1] = fmaf(v, wa1[k], acc[j][1]);
          acc[j][2] = fmaf(v, wb0[k], acc[j][2]);
          acc[j][3] = fmaf(v, wb1[k], acc[j][3]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int l = l0 + r0 + j;
      if (l >= rows_out) break;
      float a0 = acc[j][0] + ba0, a1 = acc[j][1] + ba1;
      a0 = a0 > 0.f ? a0 : a0 * slope;
      a1 = a1 > 0.f ? a1 : a1 * slope;
      float s0 = acc[j][2] + bb0, s1 = acc[j][3] + bb1;
      if (l >= valid_rows) a0 = a1 = s0 = s1 = 0.f;
      const long long row = (long long)seq * rows_out + l;
      *reinterpret_cast<float2*>(sc + row * COUT + c0) = make_float2(s0, s1);
      if (y1) *reinterpret_cast<float2*>(y1 + row * COUT + c0) = make_float2(a0, a1);
      if (P.ptr) stem_store_planes2<F16>(P, row, c0, a0, a1);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// out = LayerNorm(x + r): one warp per row, row kept in registers, two-pass mean / variance.
// ---------------------------------------------------------------------------------------------------
template <int VEC, bool F16>   // float4 chunks per lane: ch = VEC * 128; plane format
__global__ void __launch_bounds__(256) add_layernorm_kernel(
    const float* __restrict__ x, const float* __restrict__ r, const float* __restrict__ gamma,
    const float* __restrict__ beta, float* __restrict__ out, long long rows, float eps, PmPlanes P) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  constexpr int CH = VEC * 128;
  const float4* __restrict__ xr = reinterpret_cast<const float4*>(x + row * CH);
  const float4* __restrict__ rr = r ? reinterpret_cast<const float4*>(r + row * CH) : nullptr;
  float4 v[VEC];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    v[i] = xr[lane + 32 * i];
    if (rr) {
      const float4 t = rr[lane + 32 * i];
      v[i].x += t.x; v[i].y += t.y; v[i].z += t.z; v[i].w += t.w;
    }
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float mean = pm_warp_sum(s) * (1.f / CH);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float rstd = rsqrtf(pm_warp_sum(q) * (1.f / CH) + eps);
  const float4* __restrict__ g4 = reinterpret_cast<const float4*>(gamma);
  const float4* __restrict__ b4 = reinterpret_cast<const float4*>(beta);
  float4* __restrict__ o4 = out ? reinterpret_cast<float4*>(out + row * CH) : nullptr;
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const float4 g = g4[lane + 32 * i], bb = b4[lane + 32 * i];
    float4 o;
    o.x = (v[i].x - mean) * rstd * g.x + bb.x;
    o.y = (v[i].y - mean) * rstd * g.y + bb.y;
    o.z = (v[i].z - mean) * rstd * g.z + bb.z;
    o.w = (v[i].w - mean) * rstd * g.w + bb.w;
    if (o4) o4[lane + 32 * i] = o;
    if (P.ptr) pm_store_planes4_t<F16>(P, row, (lane + 32 * i) * 4, o);
  }
}

// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 pick_row(int code, const float* pe, const float* spk, int b, int t, int ch, int c4) {
  if (code == 1) return reinterpret_cast<const float4*>(pe + (long long)t * ch)[c4];
  if (code == 2) return reinterpret_cast<const float4*>(spk + (long long)b * ch)[c4];
  return make_float4(0.f, 0.f, 0.f, 0.f);
}

template <bool F16>
__global__ void __launch_bounds__(256) add_rows_kernel(
    const float* __restrict__ x, const float* __restrict__ pe, const float* __restrict__ spk,
    int first, int second, float* __restrict__ out, int batch, int rows, int ch, PmPlanes P) {
  const int ch4 = ch >> 2;
  const long long total = (long long)batch * rows * ch4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c4 = (int)(i % ch4);
    const long long bt = i / ch4;
    const int t = (int)(bt % rows), b = (int)(bt / rows);
    float4 v = x ? reinterpret_cast<const float4*>(x)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    if (first) {
      const float4 a = pick_row(first, pe, spk, b, t, ch, c4);
      v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
    }
    if (second) {
      const float4 a = pick_row(second, pe, spk, b, t, ch, c4);
      v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
    }
    if (out) reinterpret_cast<float4*>(out)[i] = v;
    if (P.ptr) pm_store_planes4_t<F16>(P, bt, c4 * 4, v);
  }
}

// rows x ch (ch % 4 == 0 when planes are requested; otherwise the tensor is treated as one flat row)
template <bool F16>
__global__ void __launch_bounds__(256) add2_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                   float* __restrict__ out, long long n4, long long n, int ch4,
                                                   PmPlanes P) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
       i += (long long)gridDim.x * blockDim.x) {
    const float4 u = reinterpret_cast<const float4*>(a)[i], v = reinterpret_cast<const float4*>(b)[i];
    const float4 o = make_float4(u.x + v.x, u.y + v.y, u.z + v.z, u.w + v.w);
    if (out) reinterpret_cast<float4*>(out)[i] = o;
    if (P.ptr) pm_store_planes4_t<F16>(P, i / ch4, (int)(i % ch4) * 4, o);
  }
  // scalar tail (n not a multiple of 4; never with planes)
  if (blockIdx.x == 0 && out) {
    for (long long i = n4 * 4 + threadIdx.x; i < n; i += blockDim.x) out[i] = a[i] + b[i];
  }
}

template <bool F16>
__global__ void __launch_bounds__(256) window_input_kernel(
    const float* __restrict__ motion, const float* __restrict__ mask, const float* __restrict__ seed,
    const float* __restrict__ mask_embedding, float* __restrict__ out,
    int batch, int total_len, int start, int win_len, int pre, int ch, long long seed_bs, PmPlanes P,
    const int* __restrict__ win_len_valid) {
  const long long total = (long long)batch * win_len * ch;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % ch);
    const long long bf = i / ch;
    const int f = (int)(bf % win_len), b = (int)(bf / win_len);
    const long long src = ((long long)b * total_len + start + f) * ch + c;
    // defaults of inference() when the caller passes no masked_motion / mask (M.py:369-377): identity rotations in
    // rot6d ([1,0,0,0,1,0] per joint) + zero trans / contact, everything masked
    float m = mask ? mask[src] : 1.f;
    float v = motion ? motion[src] : ((c < ch - 7 && (c % 6 == 0 || c % 6 == 4)) ? 1.f : 0.f);
    if (f < pre) {                    // M.py:386-391
      if (m != 0.f && seed) v = seed[(long long)b * seed_bs + (long long)f * ch + c];   // no seed yet (first window): motion itself, M.py:379
      m = 0.f;
    }
    float o = (m == 1.f) ? mask_embedding[c] : v;   // M.py:267-268
    if (win_len_valid && f >= __ldg(win_len_valid + b)) o = 0.f;     // ragged batch: zero rows beyond the clip's window
    if (out) out[i] = o;
    if (P.ptr) pm_store_planes_t<F16>(P, bf, c, o);
  }
}

inline int grid_for(long long work, int threads) {
  long long g = (work + threads - 1) / threads;
  const long long cap = 148LL * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace

static int wav_stem_run(const float* audio, long long a_bs, long long a_ws, int batch, int windows,
                        int n_samples, const float* w1, const float* b1, const float* wd,
                        const float* bd, int cout, int ksize, int stride, int pad, int rows_out,
                        float slope, float* y1, float* sc,
                        uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, const int* n_valid, void* stream) {
  PM_REQUIRE(audio && w1 && b1 && wd && bd && sc && (y1 || planes));
  PM_REQUIRE(batch > 0 && windows > 0 && n_samples > 0 && cout > 0 && stride > 0 && rows_out > 0);
  PM_TAKE_FMT(p_nsplit, f16);
  PM_REQUIRE(pm_planes_ok(planes, p_ps, p_ld, p_nsplit, cout, false));
  PM_REQUIRE(!planes || ((p_ld & 1) == 0 && (p_ps & 1) == 0 && (reinterpret_cast<uintptr_t>(planes) & 3) == 0));
  PM_REQUIRE((reinterpret_cast<uintptr_t>(sc) & 7) == 0 && (!y1 || (reinterpret_cast<uintptr_t>(y1) & 7) == 0));
  if (ksize != 15 || (cout != 32 && cout != 64)) return PM_EUNSUPPORTED;
  PM_REQUIRE((long long)batch * windows <= 65535);
  const size_t smem = (size_t)((STEM_ROWS - 1) * stride + ksize) * sizeof(float);
  PM_REQUIRE(smem <= 48 * 1024);
  const PmPlanes P{reinterpret_cast<__nv_bfloat16*>(planes), p_ps, p_ld, planes ? p_nsplit : 0};
  dim3 grid(pm_cdiv(rows_out, STEM_ROWS), batch * windows);
  cudaStream_t st = (cudaStream_t)stream;
#define PM_STEM(CO, F)                                                                                          \
  wav_stem_kernel<15, CO, F><<<grid, STEM_THREADS, smem, st>>>(audio, a_bs, a_ws, batch, n_samples, w1, b1, wd, bd, \
                                                               stride, pad, rows_out, slope, y1, sc, P, n_valid)
  if (cout == 64) { if (f16) PM_STEM(64, true); else PM_STEM(64, false); }
  else { if (f16) PM_STEM(32, true); else PM_STEM(32, false); }
#undef PM_STEM
  PM_LAUNCH_CHECK();
}

extern "C" int pm_wav_stem_f32(const float* audio, long long a_bs, long long a_ws, int batch, int windows,
                               int n_samples, const float* w1, const float* b1, const float* wd,
                               const float* bd, int cout, int ksize, int stride, int pad, int rows_out,
                               float slope, float* y1, float* sc,
                               uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream) {
  return wav_stem_run(audio, a_bs, a_ws, batch, windows, n_samples, w1, b1, wd, bd, cout, ksize, stride, pad, rows_out,
                      slope, y1, sc, planes, p_ps, p_ld, p_nsplit, nullptr, stream);
}

extern "C" int pm_wav_stem_rl(const float* audio, long long a_bs, long long a_ws, int batch, int windows,
                              int n_samples, const float* w1, const float* b1, const float* wd,
                              const float* bd, int cout, int ksize, int stride, int pad, int rows_out,
                              float slope, float* y1, float* sc,
                              uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, const int* n_valid, void* stream) {
  return wav_stem_run(audio, a_bs, a_ws, batch, windows, n_samples, w1, b1, wd, bd, cout, ksize, stride, pad, rows_out,
                      slope, y1, sc, planes, p_ps, p_ld, p_nsplit, n_valid, stream);
}

extern "C" int pm_add_layernorm_f32(const float* x, const float* r, const float* gamma, const float* beta,
                                    float* out, long long rows, int ch, float eps,
                                    uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream) {
  PM_REQUIRE(x && gamma && beta && (out || planes) && rows >= 0);
  PM_TAKE_FMT(p_nsplit, f16);
  PM_REQUIRE(pm_planes_ok(planes, p_ps, p_ld, p_nsplit, ch, true));
  const PmPlanes P{reinterpret_cast<__nv_bfloat16*>(planes), p_ps, p_ld, p_nsplit};
  if (rows == 0) return PM_OK;
  const int warps = 8;
  const unsigned grid = (unsigned)((rows + warps - 1) / warps);
  cudaStream_t st = (cudaStream_t)stream;
  switch (ch) {
    case 256:
      if (f16) add_layernorm_kernel<2, true><<<grid, warps * 32, 0, st>>>(x, r, gamma, beta, out, rows, eps, P);
      else add_layernorm_kernel<2, false><<<grid, warps * 32, 0, st>>>(x, r, gamma, beta, out, rows, eps, P);
      break;
    case 512:
      if (f16) add_layernorm_kernel<4, true><<<grid, warps * 32, 0, st>>>(x, r, gamma, beta, out, rows, eps, P);
      else add_layernorm_kernel<4, false><<<grid, warps * 32, 0, st>>>(x, r, gamma, beta, out, rows, eps, P);
      break;
    case 768:
      if (f16) add_layernorm_kernel<6, true><<<grid, warps * 32, 0, st>>>(x, r, gamma, beta, out, rows, eps, P);
      else add_layernorm_kernel<6, false><<<grid, warps * 32, 0, st>>>(x, r, gamma, beta, out, rows, eps, P);
      break;
    case 1024:
      if (f16) add_layernorm_kernel<8, true><<<grid, warps * 32, 0, st>>>(x, r, gamma, beta, out, rows, eps, P);
      else add_layernorm_kernel<8, false><<<grid, warps * 32, 0, st>>>(x, r, gamma, beta, out, rows, eps, P);
      break;
    default: return PM_EUNSUPPORTED;
  }
  PM_LAUNCH_CHECK();
}

extern "C" int pm_add_rows_f32(const float* x, const float* pe, const float* spk, int first, int second,
                               float* out, int batch, int rows, int ch,
                               uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream) {
  PM_REQUIRE((out || planes) && batch >= 0 && rows >= 0 && ch > 0 && (ch & 3) == 0);
  PM_TAKE_FMT(p_nsplit, f16);
  PM_REQUIRE(pm_planes_ok(planes, p_ps, p_ld, p_nsplit, ch, true));
  const PmPlanes P{reinterpret_cast<__nv_bfloat16*>(planes), p_ps, p_ld, p_nsplit};
  PM_REQUIRE(first >= 0 && first <= 2 && second >= 0 && second <= 2);
  PM_REQUIRE((first != 1 && second != 1) || pe);
  PM_REQUIRE((first != 2 && second != 2) || spk);
  const long long total = (long long)batch * rows * (ch >> 2);
  if (total == 0) return PM_OK;
  if (f16) add_rows_kernel<true><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(x, pe, spk, first, second, out,
                                                                                  batch, rows, ch, P);
  else add_rows_kernel<false><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(x, pe, spk, first, second, out,
                                                                               batch, rows, ch, P);
  PM_LAUNCH_CHECK();
}

extern "C" int pm_add2_f32(const float* a, const float* b, float* out, long long n, int ch,
                           uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream) {
  PM_REQUIRE(a && b && (out || planes) && n >= 0);
  PM_REQUIRE(!planes || (ch > 0 && (ch & 3) == 0 && n % ch == 0));
  PM_TAKE_FMT(p_nsplit, f16);
  PM_REQUIRE(pm_planes_ok(planes, p_ps, p_ld, p_nsplit, ch, true));
  const PmPlanes P{reinterpret_cast<__nv_bfloat16*>(planes), p_ps, p_ld, p_nsplit};
  if (n == 0) return PM_OK;
  if (f16) add2_kernel<true><<<grid_for(n / 4 + 1, 256), 256, 0, (cudaStream_t)stream>>>(a, b, out, n / 4, n, planes ? ch / 4 : 1, P);
  else add2_kernel<false><<<grid_for(n / 4 + 1, 256), 256, 0, (cudaStream_t)stream>>>(a, b, out, n / 4, n, planes ? ch / 4 : 1, P);
  PM_LAUNCH_CHECK();
}

static int window_input_run(const float* motion, const float* mask, const float* seed,
                            const float* mask_embedding, float* out, int batch, int total_len,
                            int start, int win_len, int pre, int ch, long long seed_bs,
                            uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, const int* win_len_valid,
                            void* stream) {
  PM_REQUIRE(mask_embedding && (out || planes));
  PM_TAKE_FMT(p_nsplit, f16);
  PM_REQUIRE(pm_planes_ok(planes, p_ps, p_ld, p_nsplit, ch, false));
  const PmPlanes P{reinterpret_cast<__nv_bfloat16*>(planes), p_ps, p_ld, p_nsplit};
  PM_REQUIRE(batch >= 0 && win_len >= 0 && start >= 0 && start + win_len <= total_len && pre >= 0 && ch > 0);
  const long long total = (long long)batch * win_len * ch;
  if (total == 0) return PM_OK;
  if (f16) window_input_kernel<true><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      motion, mask, seed, mask_embedding, out, batch, total_len, start, win_len, pre, ch, seed_bs, P, win_len_valid);
  else window_input_kernel<false><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
      motion, mask, seed, mask_embedding, out, batch, total_len, start, win_len, pre, ch, seed_bs, P, win_len_valid);
  PM_LAUNCH_CHECK();
}

extern "C" int pm_window_input_f32(const float* motion, const float* mask, const float* seed,
                                   const float* mask_embedding, float* out, int batch, int total_len,
                                   int start, int win_len, int pre, int ch, long long seed_bs,
                                   uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, void* stream) {
  return window_input_run(motion, mask, seed, mask_embedding, out, batch, total_len, start, win_len, pre, ch, seed_bs,
                          planes, p_ps, p_ld, p_nsplit, nullptr, stream);
}

extern "C" int pm_window_input_rl(const float* motion, const float* mask, const float* seed,
                                  const float* mask_embedding, float* out, int batch, int total_len,
                                  int start, int win_len, int pre, int ch, long long seed_bs,
                                  uint16_t* planes, long long p_ps, int p_ld, int p_nsplit, const int* win_len_valid,
                                  void* stream) {
  return window_input_run(motion, mask, seed, mask_embedding, out, batch, total_len, start, win_len, pre, ch, seed_bs,
                          planes, p_ps, p_ld, p_nsplit, win_len_valid, stream);
}
