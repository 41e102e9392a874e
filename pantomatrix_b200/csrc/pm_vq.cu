// VQ codebook kernels: fused L2-argmin lookup, row argmax, codebook gather.
// Contracts and reference call sites: include/pm_emage.h.
#include "pm_common.cuh"
#include "../../include/pm_emage.h"

namespace {

constexpr int ED = 256;          // e_dim
constexpr int EDP = ED + 1;      // padded smem row
constexpr int RT = 64;           // rows per CTA
constexpr int CT = 64;           // codes per chunk
constexpr int NT = 256;

// d(r,k) = (|z_r|^2 + |e_k|^2) - 2 z_r.e_k in fp32 (same expression as M.py:64), argmin with the
// lowest index winning ties (torch.argmin).  The dot products are the hot part: a 64x64x256 register-
// tiled product per chunk, z tile resident in smem, codebook (256 KB) streamed from L2 in 64 KB chunks.
__global__ void __launch_bounds__(NT) l2_argmin_kernel(
    const float* __restrict__ z, long long rows, int rows_per_batch, long long z_bs, const float* __restrict__ codebook,
    const float* __restrict__ e2, int n_codes, long long* __restrict__ index) {
  extern __shared__ float smem[];
  float* Zs = smem;                 // [RT][EDP]
  float* Es = Zs + RT * EDP;        // [CT][EDP]
  float* z2s = Es + CT * EDP;       // [RT]
  const int tid = threadIdx.x;
  const long long r0 = (long long)blockIdx.x * RT;

  for (int i = tid; i < RT * (ED / 4); i += NT) {          // coalesced float4 loads of the z tile
    const int r = i / (ED / 4), c4 = i % (ED / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r0 + r < rows) {
      const unsigned g = (unsigned)(r0 + r), gb = g / (unsigned)rows_per_batch;      // strided views are small (host checks)
      const float* zr = rows_per_batch == 0x7fffffff ? z + (r0 + r) * ED
                                                     : z + (long long)gb * z_bs + (long long)(g - gb * (unsigned)rows_per_batch) * ED;
      v = *reinterpret_cast<const float4*>(zr + c4 * 4);
    }
    float* d = Zs + r * EDP + c4 * 4;
    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
  }
  __syncthreads();
  {
    const int warp = tid >> 5, lane = tid & 31;
    for (int r = warp; r < RT; r += NT / 32) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < ED / 32; ++i) { const float v = Zs[r * EDP + lane + 32 * i]; s = fmaf(v, v, s); }
      s = pm_warp_sum(s);
      if (lane == 0) z2s[r] = s;
    }
  }

  const int ti = tid >> 4, tj = tid & 15;
  float best[4];
  int bestk[4];
#pragma unroll
  for (int a = 0; a < 4; ++a) { best[a] = INFINITY; bestk[a] = 0x7fffffff; }   // 0x7fffffff = nothing yet (NaN rows: see the end)

  for (int k0 = 0; k0 < n_codes; k0 += CT) {
    __syncthreads();                                        // previous chunk fully consumed (and z2s visible)
    for (int i = tid; i < CT * (ED / 4); i += NT) {
      const int r = i / (ED / 4), c4 = i % (ED / 4);
      const float4 v = *reinterpret_cast<const float4*>(codebook + (long long)(k0 + r) * ED + c4 * 4);
      float* d = Es + r * EDP + c4 * 4;
      d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
    __syncthreads();
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[a][c] = 0.f;
    const float* zp = Zs + (ti * 4) * EDP;
    const float* ep = Es + (tj * 4) * EDP;
#pragma unroll 4
    for (int d = 0; d < ED; ++d) {
      float zv[4], ev[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) { zv[a] = zp[a * EDP + d]; ev[a] = ep[a * EDP + d]; }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][c] = fmaf(zv[a], ev[c], acc[a][c]);
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int k = k0 + tj * 4 + c;
      const float ek = __ldg(e2 + k);
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const float dist = __fsub_rn(__fadd_rn(z2s[ti * 4 + a], ek), __fmul_rn(2.f, acc[a][c]));
        if (dist < best[a] || (dist == best[a] && k < bestk[a])) { best[a] = dist; bestk[a] = k; }
      }
    }
  }
  // combine the 16 lanes (tj) that share a row group; they are 16 consecutive lanes of one warp
#pragma unroll
  for (int a = 0; a < 4; ++a) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best[a], o);
      const int ok = __shfl_xor_sync(0xffffffffu, bestk[a], o);
      if (ob < best[a] || (ob == best[a] && ok < bestk[a])) { best[a] = ob; bestk[a] = ok; }
    }
    const long long r = r0 + ti * 4 + a;
    // a row whose distances are all NaN never updates bestk: emit 0, the index torch.argmin returns for it
    if (tj == 0 && r < rows) index[r] = bestk[a] == 0x7fffffff ? 0 : bestk[a];
  }
}

constexpr size_t kL2Smem = (size_t)(RT * EDP + CT * EDP + RT) * sizeof(float);

__global__ void __launch_bounds__(256) row_argmax_kernel(const float* __restrict__ x, long long rows, int ch,
                                                         int ldx, int rows_per_batch, long long x_bs,
                                                         long long* __restrict__ index, int* __restrict__ nonfinite) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const unsigned rb = (unsigned)row / (unsigned)rows_per_batch;            // strided views are small (host checks)
  const float* __restrict__ xr = rows_per_batch == 0x7fffffff ? x + row * ldx
                                                              : x + (long long)rb * x_bs + (long long)((unsigned)row - rb * (unsigned)rows_per_batch) * ldx;
  float best = -INFINITY;
  int bk = 0x7fffffff;
  bool bad = false;
  for (int c = lane; c < ch; c += 32) {        // increasing c per lane: strict > keeps the first max
    const float v = xr[c];
    bad |= !isfinite(v);
    if (v > best || bk == 0x7fffffff) { best = v; bk = c; }
  }
  if (nonfinite && __any_sync(0xffffffffu, bad) && lane == 0) atomicExch(nonfinite, 1);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int ok = __shfl_xor_sync(0xffffffffu, bk, o);
    if (ob > best || (ob == best && ok < bk)) { best = ob; bk = ok; }
  }
  if (lane == 0) index[row] = bk;
}

template <bool F16>
__global__ void __launch_bounds__(256) gather_rows_kernel(const float* __restrict__ codebook, long long n_table,
                                                          const long long* __restrict__ index, long long rows,
                                                          int ch4, float* __restrict__ out, PmPlanes P,
                                                          const int* __restrict__ row_limit, int rows_per_clip) {
  const long long total = rows * ch4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / ch4;
    const int c4 = (int)(i % ch4);
    long long k = index[r];                       // out-of-range ids (user input) are clamped: never read outside the table
    k = k < 0 ? 0 : (k >= n_table ? n_table - 1 : k);
    float4 v = reinterpret_cast<const float4*>(codebook)[k * ch4 + c4];
    if (row_limit && r % rows_per_clip >= __ldg(row_limit + r / rows_per_clip)) v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (out) reinterpret_cast<float4*>(out)[i] = v;
    if (P.ptr) pm_store_planes4_t<F16>(P, r, c4 * 4, v);
  }
}

__global__ void __launch_bounds__(256) row_sqnorm_kernel(const float* __restrict__ x, int rows, int ch,
                                                         float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  float s = 0.f;
  for (int c = lane; c < ch; c += 32) { const float v = x[(long long)row * ch + c]; s = fmaf(v, v, s); }
  s = pm_warp_sum(s);
  if (lane == 0) out[row] = s;
}

}  // namespace

extern "C" int pm_l2_argmin_simt_f32(const float* z, long long rows, int rows_per_batch, long long z_bs,
                                     const float* codebook, const float* e2,
                                     int n_codes, int e_dim, long long* index, void* stream) {
  PM_REQUIRE(z && codebook && e2 && index && rows >= 0);
  if (rows_per_batch <= 0 || z_bs == (long long)rows_per_batch * ED) { rows_per_batch = 0x7fffffff; z_bs = 0; }
  PM_REQUIRE((z_bs & 3) == 0 && (rows_per_batch == 0x7fffffff || rows < 0x7fffffffLL));
  if (e_dim != ED || n_codes <= 0 || n_codes % CT != 0) return PM_EUNSUPPORTED;
  if (rows == 0) return PM_OK;
  {   // per device, cheap: no process-wide "configured" flag (a second GPU in the same process needs it too)
    cudaError_t e = cudaFuncSetAttribute(l2_argmin_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kL2Smem);
    if (e != cudaSuccess) return (int)e;
  }
  const long long grid = (rows + RT - 1) / RT;
  PM_REQUIRE(grid <= 0x7fffffffLL);
  l2_argmin_kernel<<<(unsigned)grid, NT, kL2Smem, (cudaStream_t)stream>>>(z, rows, rows_per_batch, z_bs, codebook, e2, n_codes, index);
  PM_LAUNCH_CHECK();
}

extern "C" int pm_l2_argmin_f32(const float* z, long long rows, int rows_per_batch, long long z_bs,
                                const float* codebook, const float* e2,
                                int n_codes, int e_dim, long long* index, void* stream) {
  // 256 codes x 256 dims (every EMAGE codebook): tensor-core screen + exact fp32 re-scoring (pm_vq_tc.cu);
  // other codebook sizes: the fp32 SIMT kernel above.  Both return the fp32 argmin with first-index ties.
  if (n_codes == 256 && e_dim == 256 && z && codebook && (reinterpret_cast<uintptr_t>(z) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(codebook) & 15) == 0)
    return pm_l2_argmin_tc(z, rows, rows_per_batch, z_bs, codebook, e2, n_codes, e_dim, index, 0, stream);
  return pm_l2_argmin_simt_f32(z, rows, rows_per_batch, z_bs, codebook, e2, n_codes, e_dim, index, stream);
}

extern "C" int pm_row_argmax_f32(const float* x, long long rows, int ch, int ldx, int rows_per_batch, long long x_bs,
                                 long long* index, int* nonfinite, void* stream) {
  PM_REQUIRE(x && index && rows >= 0 && ch > 0 && ldx >= ch);
  if (rows == 0) return PM_OK;
  if (rows_per_batch <= 0 || x_bs == (long long)rows_per_batch * ldx) { rows_per_batch = 0x7fffffff; x_bs = 0; }   // dense (rows, ldx)
  PM_REQUIRE(rows_per_batch == 0x7fffffff || rows < 0x7fffffffLL);
  row_argmax_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(x, rows, ch, ldx, rows_per_batch, x_bs,
                                                                                  index, nonfinite);
  PM_LAUNCH_CHECK();
}

static int gather_rows_run(const float* codebook, long long n_table, const long long* index, long long rows, int ch,
                           float* out, uint16_t* planes, long long p_ps, int p_ld, int p_nsplit,
                           const int* row_limit, int rows_per_clip, void* stream) {
  PM_REQUIRE(codebook && index && (out || planes) && rows >= 0 && n_table > 0 && ch > 0 && (ch & 3) == 0);
  PM_REQUIRE(!row_limit || rows_per_clip > 0);
  PM_TAKE_FMT(p_nsplit, f16);
  PM_REQUIRE(pm_planes_ok(planes, p_ps, p_ld, p_nsplit, ch, true));
  const PmPlanes P{reinterpret_cast<__nv_bfloat16*>(planes), p_ps, p_ld, p_nsplit};
  if (rows == 0) return PM_OK;
  long long g = (rows * (ch >> 2) + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  if (f16) gather_rows_kernel<true><<<(unsigned)g, 256, 0, (cudaStream_t)stream>>>(codebook, n_table, index, rows, ch >> 2, out, P,
                                                                                   row_limit, rows_per_clip);
  else gather_rows_kernel<false><<<(unsigned)g, 256, 0, (cudaStream_t)stream>>>(codebook, n_table, index, rows, ch >> 2, out, P,
                                                                                 row_limit, rows_per_clip);
  PM_LAUNCH_CHECK();
}

extern "C" int pm_gather_rows_f32(const float* codebook, long long n_table, const long long* index, long long rows, int ch,
                                  float* out, uint16_t* planes, long long p_ps, int p_ld, int p_nsplit,
                                  void* stream) {
  return gather_rows_run(codebook, n_table, index, rows, ch, out, planes, p_ps, p_ld, p_nsplit, nullptr, 0, stream);
}

extern "C" int pm_gather_rows_rl(const float* codebook, long long n_table, const long long* index, long long rows, int ch,
                                 float* out, uint16_t* planes, long long p_ps, int p_ld, int p_nsplit,
                                 const int* row_limit, int rows_per_clip, void* stream) {
  return gather_rows_run(codebook, n_table, index, rows, ch, out, planes, p_ps, p_ld, p_nsplit, row_limit, rows_per_clip,
                         stream);
}

extern "C" int pm_row_sqnorm_f32(const float* x, int rows, int ch, float* out, void* stream) {
  PM_REQUIRE(x && out && rows >= 0 && ch > 0);
  if (rows == 0) return PM_OK;
  row_sqnorm_kernel<<<(rows + 7) / 8, 256, 0, (cudaStream_t)stream>>>(x, rows, ch, out);
  PM_LAUNCH_CHECK();
}
