// Direct convolution for layers whose input has very few channels (Cin <= 4): the 1-channel nnU-Net stem
// (encoder.stages.0.0.convs.0, built at models/seg_model.py:174-191) and the 2-channel FLAVR stem
// k(3,7,7) s(1,2,2) (models/FLAVR/resnet_3D.py:42-50).  K = taps*Cin is 27..294, far too thin to feed the
// tensor cores from an NDHWC tile (Cin would have to be padded 8-16x), and the layer is HBM-bound anyway
// (SURVEY.md section 7.3, enc0.0: 26 FLOP/B): the input is read as the caller hands it (NCDHW f32,
// train_all.py:524), weights live in shared memory, each thread produces one output voxel x 16 channels and
// writes NDHWC bf16 so the next layer's TMA tiles are ready-made.
#include "engine.h"
#include "ptx.cuh"

#include <cuda_bf16.h>

#include <algorithm>

namespace rehr {

// tensor-core stem (stem_mma.cu): Cin = 1, Cout = 32, k3 s1 p1
bool stem_mma_supported(int cin, int cout, int wd);
size_t stem_mma_wgrad_workspace();
int launch_stem_fwd_mma(const float* x, const float* w, const float* bias, __nv_bfloat16* y, long long ldy, int y_f16, int n, int d, int h, int wd,
                        int act, float slope, int planar, cudaStream_t stream);
int launch_stem_wgrad_mma(const float* x, const __nv_bfloat16* dy, long long lddy, int n, int d, int h, int wd, float* dw, int accumulate,
                          float* ws, int planar, cudaStream_t stream);

static constexpr int kScMaxCin = 4;
static constexpr int kScCoutPerThread = 16;

struct SmallCinArgs {
  const float* x;      // [n][cin][d][h][w]
  const float* w;      // [cout][cin][T]
  const float* bias;   // [cout] or null
  __nv_bfloat16* y;    // NDHWC
  long long ldy;
  int n, cin, d, h, wd;     // input dims
  int od, oh, ow, cout;     // output dims
  int kd, kh, kw, sd, sh, sw, pd, ph, pw;
  int act;
  float slope;
  int y_f16;           // storage format of y (rehr_dtype)
  RangeSlot* range;    // fp16 saturation record of y (rehr_range_sink), null = not checked
};

// weights in smem as [cin*T][cout] (cout fastest) so that a thread's 16 channels are 4 float4 broadcasts.
__global__ void __launch_bounds__(256) smallcin_fwd_kernel(const SmallCinArgs a) {
  extern __shared__ float sw[];
  const int T = a.kd * a.kh * a.kw;
  const int KT = a.cin * T;
  for (int i = threadIdx.x; i < KT * a.cout; i += blockDim.x) {
    const int co = i % a.cout, k = i / a.cout;  // k = ci*T + t
    sw[i] = a.w[(long long)co * KT + k];
  }
  __syncthreads();
  const int cgroups = (a.cout + kScCoutPerThread - 1) / kScCoutPerThread;
  const long long ovox = (long long)a.n * a.od * a.oh * a.ow;
  const long long items = ovox * cgroups;
  const long long in_plane = (long long)a.h * a.wd, in_vol = in_plane * a.d;
  for (long long it = blockIdx.x * (long long)blockDim.x + threadIdx.x; it < items; it += (long long)gridDim.x * blockDim.x) {
    // consecutive threads -> consecutive output voxels along w (coalesced input reads); channel group outermost
    const int cg = (int)(it / ovox);
    long long v = it % ovox;
    const int ox = (int)(v % a.ow);
    long long r = v / a.ow;
    const int oy = (int)(r % a.oh);
    r /= a.oh;
    const int oz = (int)(r % a.od);
    const int nn = (int)(r / a.od);
    const int c0 = cg * kScCoutPerThread;
    float acc[kScCoutPerThread];
#pragma unroll
    for (int i = 0; i < kScCoutPerThread; ++i) acc[i] = (a.bias && c0 + i < a.cout) ? a.bias[c0 + i] : 0.f;
    for (int ci = 0; ci < a.cin; ++ci) {
      const float* xp = a.x + ((long long)nn * a.cin + ci) * in_vol;
      for (int kz = 0; kz < a.kd; ++kz) {
        const int iz = oz * a.sd + kz - a.pd;
        if (iz < 0 || iz >= a.d) continue;
        for (int ky = 0; ky < a.kh; ++ky) {
          const int iy = oy * a.sh + ky - a.ph;
          if (iy < 0 || iy >= a.h) continue;
          for (int kx = 0; kx < a.kw; ++kx) {
            const int ix = ox * a.sw + kx - a.pw;
            if (ix < 0 || ix >= a.wd) continue;
            const float xv = __ldg(xp + iz * in_plane + (long long)iy * a.wd + ix);
            const float* wp = sw + (size_t)(ci * T + (kz * a.kh + ky) * a.kw + kx) * a.cout + c0;
            if (c0 + kScCoutPerThread <= a.cout) {
#pragma unroll
              for (int i = 0; i < kScCoutPerThread; i += 4) {
                const float4 w4 = *reinterpret_cast<const float4*>(wp + i);
                acc[i] = fmaf(xv, w4.x, acc[i]);
                acc[i + 1] = fmaf(xv, w4.y, acc[i + 1]);
                acc[i + 2] = fmaf(xv, w4.z, acc[i + 2]);
                acc[i + 3] = fmaf(xv, w4.w, acc[i + 3]);
              }
            } else {
              for (int i = 0; i < kScCoutPerThread; ++i)
                if (c0 + i < a.cout) acc[i] = fmaf(xv, wp[i], acc[i]);
            }
          }
        }
      }
    }
    __nv_bfloat16* o = a.y + v * a.ldy + c0;
    if (c0 + kScCoutPerThread <= a.cout) {
      uint4 lo, hi;
      float f[kScCoutPerThread];
#pragma unroll
      for (int i = 0; i < kScCoutPerThread; ++i) {
        float z = acc[i];
        if (a.act == REHR_ACT_RELU) z = z > 0.f ? z : 0.f;
        if (a.act == REHR_ACT_LRELU) z = z > 0.f ? z : z * a.slope;
        f[i] = z;
      }
      if (a.range != nullptr) range_check<kScCoutPerThread>(a.range, f);
      uint32_t* l2 = reinterpret_cast<uint32_t*>(&lo);
      uint32_t* h2 = reinterpret_cast<uint32_t*>(&hi);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        l2[i] = pack16x2(f[2 * i], f[2 * i + 1], a.y_f16);
        h2[i] = pack16x2(f[8 + 2 * i], f[8 + 2 * i + 1], a.y_f16);
      }
      reinterpret_cast<uint4*>(o)[0] = lo;
      reinterpret_cast<uint4*>(o)[1] = hi;
    } else {
      for (int i = 0; i < kScCoutPerThread; ++i)
        if (c0 + i < a.cout) {
          float z = acc[i];
          if (a.act == REHR_ACT_RELU) z = z > 0.f ? z : 0.f;
          if (a.act == REHR_ACT_LRELU) z = z > 0.f ? z : z * a.slope;
          reinterpret_cast<unsigned short*>(o)[i] = pack16(z, a.y_f16);
          acc[i] = z;
        }
      if (a.range != nullptr) range_check<kScCoutPerThread>(a.range, acc, a.cout - c0);
    }
  }
}

// Fast forward path for k = 3x3x3, stride 1, pad 1, Cout = 32 (the nnU-Net stem at the C1 size: 4.2 M voxels): a CTA stages the
// CIN x 3 x 10 x (W+2) fp32 input rows that 8 output rows (one per warp) need plus the 27*CIN x 32 weights in shared memory; a
// thread owns one output voxel and all 32 channels, so the inner loop is fully unrolled (no bounds tests, no index arithmetic),
// every x value is one conflict-free shared load, weights are float4 broadcasts, and a warp writes 2 KB of contiguous NDHWC bf16.
template <int CIN>
__global__ void __launch_bounds__(256) smallcin_fwd_k3c32_kernel(const SmallCinArgs a) {
  extern __shared__ float sm[];  // [CIN*27][32] weights, then [CIN][3][10][Wa] input rows
  const int Wa = a.wd + 2;
  float* sw = sm;
  float* sx = sm + CIN * 27 * 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < CIN * 27 * 32; i += 256) {
    const int co = i % 32, k = i / 32;  // k = ci*27 + t
    sw[i] = a.w[(long long)co * CIN * 27 + k];
  }
  float bias[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) bias[i] = a.bias ? __ldg(a.bias + i) : 0.f;
  const int ytiles = (a.oh + 7) / 8;
  const long long tiles = (long long)a.n * a.od * ytiles;
  const long long in_plane = (long long)a.h * a.wd, in_vol = in_plane * a.d;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int yt = (int)(tile % ytiles);
    long long r = tile / ytiles;
    const int oz = (int)(r % a.od);
    const int nn = (int)(r / a.od);
    const int oy0 = yt * 8;
    __syncthreads();
    for (int i = threadIdx.x; i < CIN * 30 * Wa; i += 256) {
      const int xx = i % Wa;
      int q = i / Wa;
      const int yy = q % 10;
      q /= 10;
      const int kz = q % 3, ci = q / 3;
      const int iz = oz + kz - 1, iy = oy0 + yy - 1, ix = xx - 1;
      float v = 0.f;
      if (iz >= 0 && iz < a.d && iy >= 0 && iy < a.h && ix >= 0 && ix < a.wd)
        v = __ldg(a.x + ((long long)nn * CIN + ci) * in_vol + iz * in_plane + (long long)iy * a.wd + ix);
      sx[i] = v;
    }
    __syncthreads();
    const int oy = oy0 + warp;
    if (oy >= a.oh) continue;
    for (int ox = lane; ox < a.ow; ox += 32) {
      // compiler barrier: without it the 27*CIN*32 loop-invariant weight loads are hoisted out of this loop into 864+
      // "registers" that ptxas spills to local memory (9.6 KB stack frame, 6x slower)
      asm volatile("" ::: "memory");
      float acc[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[i] = bias[i];
#pragma unroll
      for (int ci = 0; ci < CIN; ++ci)
#pragma unroll
        for (int kz = 0; kz < 3; ++kz)
#pragma unroll
          for (int ky = 0; ky < 3; ++ky) {
            const float* xr = sx + ((ci * 3 + kz) * 10 + warp + ky) * Wa + ox;
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
              const float xv = xr[kx];
              const float4* wp = reinterpret_cast<const float4*>(sw + (ci * 27 + (kz * 3 + ky) * 3 + kx) * 32);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float4 w4 = wp[i];
                acc[4 * i] = fmaf(xv, w4.x, acc[4 * i]);
                acc[4 * i + 1] = fmaf(xv, w4.y, acc[4 * i + 1]);
                acc[4 * i + 2] = fmaf(xv, w4.z, acc[4 * i + 2]);
                acc[4 * i + 3] = fmaf(xv, w4.w, acc[4 * i + 3]);
              }
            }
          }
      const long long v = (((long long)nn * a.od + oz) * a.oh + oy) * a.ow + ox;
      uint4* o = reinterpret_cast<uint4*>(a.y + v * a.ldy);
      uint32_t cnt = 0, mbits = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint4 u;
        uint32_t* h2 = reinterpret_cast<uint32_t*>(&u);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float z0 = acc[8 * j + 2 * i], z1 = acc[8 * j + 2 * i + 1];
          if (a.act == REHR_ACT_RELU) { z0 = z0 > 0.f ? z0 : 0.f; z1 = z1 > 0.f ? z1 : 0.f; }
          if (a.act == REHR_ACT_LRELU) { z0 = z0 > 0.f ? z0 : z0 * a.slope; z1 = z1 > 0.f ? z1 : z1 * a.slope; }
          h2[i] = pack16x2(z0, z1, a.y_f16);
          if (a.range != nullptr) { range_fold(z0, cnt, mbits); range_fold(z1, cnt, mbits); }
        }
        o[j] = u;
      }
      if (a.range != nullptr) range_flush(a.range, cnt, mbits);
    }
  }
}

template <int CIN>
static int launch_smallcin_fwd_k3c32(const SmallCinArgs& a, cudaStream_t stream) {
  const size_t smem = ((size_t)CIN * 27 * 32 + (size_t)CIN * 30 * (a.wd + 2)) * sizeof(float);
  if (smem > 200 * 1024) return REHR_UNSUPPORTED;
  static size_t attr_smem = 0;
  if (smem > 48 * 1024 && smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(smallcin_fwd_k3c32_kernel<CIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      g_last_cuda_error = (int)e;
      return REHR_CUDA_ERROR;
    }
    attr_smem = smem;
  }
  const long long tiles = (long long)a.n * a.od * ((a.oh + 7) / 8);
  const int blocks = (int)std::max<long long>(1, std::min<long long>(tiles, (long long)sm_count() * 4));
  smallcin_fwd_k3c32_kernel<CIN><<<blocks, 256, smem, stream>>>(a);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

// ------------------------------------------------------------------------------------------------
// Weight gradient: dw[co][ci][t] = sum_o dy[o, co] * x[ci, o*s + t - p].
// Warp = a run of output voxels, lane = output channel (coalesced 64 B dy rows); each lane keeps kWgAcc
// (ci, tap) accumulators in registers; layers with more than kWgAcc (ci, tap) pairs make several passes
// (blockIdx.y).  Per-block partials go to the workspace [pass][block][kWgAcc][cout] and a second kernel
// reduces them in a fixed order (deterministic).
// ------------------------------------------------------------------------------------------------
static constexpr int kWgAcc = 27;
static constexpr int kWgBlocks = 592;  // 4 x 148

struct SmallCinWgradArgs {
  const float* x;
  const __nv_bfloat16* dy;
  long long lddy;
  float* ws;
  int n, cin, d, h, wd, od, oh, ow, cout;
  int kd, kh, kw, sd, sh, sw, pd, ph, pw;
};

__global__ void __launch_bounds__(256) smallcin_wgrad_kernel(const SmallCinWgradArgs a) {
  __shared__ float red[8][kWgAcc][32];
  const int T = a.kd * a.kh * a.kw, KT = a.cin * T;
  const int pass = blockIdx.y;
  const int k0 = pass * kWgAcc;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long ovox = (long long)a.n * a.od * a.oh * a.ow;
  const long long in_plane = (long long)a.h * a.wd, in_vol = in_plane * a.d;
  const int cblocks = (a.cout + 31) / 32;
  for (int cb = 0; cb < cblocks; ++cb) {
    const int co = cb * 32 + lane;
    float acc[kWgAcc];
#pragma unroll
    for (int i = 0; i < kWgAcc; ++i) acc[i] = 0.f;
    for (long long v = (long long)blockIdx.x * 8 + warp; v < ovox; v += (long long)gridDim.x * 8) {
      const float g = co < a.cout ? __bfloat162float(a.dy[v * a.lddy + co]) : 0.f;
      const int ox = (int)(v % a.ow);
      long long r = v / a.ow;
      const int oy = (int)(r % a.oh);
      r /= a.oh;
      const int oz = (int)(r % a.od);
      const int nn = (int)(r / a.od);
#pragma unroll
      for (int i = 0; i < kWgAcc; ++i) {
        const int k = k0 + i;
        if (k < KT) {
          const int ci = k / T, t = k % T;
          const int kx = t % a.kw, ky = (t / a.kw) % a.kh, kz = t / (a.kw * a.kh);
          const int iz = oz * a.sd + kz - a.pd, iy = oy * a.sh + ky - a.ph, ix = ox * a.sw + kx - a.pw;
          if (iz >= 0 && iz < a.d && iy >= 0 && iy < a.h && ix >= 0 && ix < a.wd)
            acc[i] = fmaf(g, __ldg(a.x + ((long long)nn * a.cin + ci) * in_vol + iz * in_plane + (long long)iy * a.wd + ix), acc[i]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < kWgAcc; ++i) red[warp][i][lane] = acc[i];
    __syncthreads();
    for (int i = threadIdx.x; i < kWgAcc * 32; i += blockDim.x) {
      const int k = i / 32, l = i % 32;
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) s += red[w][k][l];
      if (cb * 32 + l < a.cout)
        a.ws[(((long long)pass * gridDim.x + blockIdx.x) * kWgAcc + k) * a.cout + cb * 32 + l] = s;
    }
    __syncthreads();
  }
}

// Fast path for k = 3x3x3, stride 1, pad 1 (the nnU-Net stem, 4.2 M voxels x 32 channels at the C1 size): the layer is
// bound by streaming dy once (268 MB bf16), so the work is organised around that stream.  A CTA stages the 3 x 10 x (W+2)
// fp32 input rows that 8 output rows (one per warp) need into shared memory; lane = output channel, so a voxel's dy row
// is one coalesced 64 B load and every x value is a shared-memory broadcast; a thread walks its row 4 voxels at a time
// (6 x values feed 12 FMAs) and keeps the CIN*27 per-channel accumulators in registers across all its tiles.  Same
// workspace layout / second-stage reduction as the generic kernel above.
template <int CIN>
__global__ void __launch_bounds__(256) smallcin_wgrad_k3_kernel(const SmallCinWgradArgs a) {
  extern __shared__ float sx[];  // [CIN][3][10][Wa] then reused as red[8][27][32]
  const int Wa = a.wd + 6;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int co = blockIdx.y * 32 + lane;
  const bool cok = co < a.cout;
  float acc[CIN * 27];
#pragma unroll
  for (int i = 0; i < CIN * 27; ++i) acc[i] = 0.f;
  const int ytiles = (a.oh + 7) / 8;
  const long long tiles = (long long)a.n * a.od * ytiles;
  const long long in_plane = (long long)a.h * a.wd, in_vol = in_plane * a.d;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int yt = (int)(tile % ytiles);
    long long r = tile / ytiles;
    const int oz = (int)(r % a.od);
    const int nn = (int)(r / a.od);
    const int oy0 = yt * 8;
    __syncthreads();
    for (int i = threadIdx.x; i < CIN * 30 * Wa; i += 256) {
      const int xx = i % Wa;
      int q = i / Wa;
      const int yy = q % 10;
      q /= 10;
      const int kz = q % 3, ci = q / 3;
      const int iz = oz + kz - 1, iy = oy0 + yy - 1, ix = xx - 1;
      float v = 0.f;
      if (iz >= 0 && iz < a.d && iy >= 0 && iy < a.h && ix >= 0 && ix < a.wd)
        v = __ldg(a.x + ((long long)nn * CIN + ci) * in_vol + iz * in_plane + (long long)iy * a.wd + ix);
      sx[i] = v;
    }
    __syncthreads();
    const int oy = oy0 + warp;
    if (oy < a.oh) {
      const __nv_bfloat16* dyrow = a.dy + ((((long long)nn * a.od + oz) * a.oh + oy) * a.ow) * a.lddy + co;
      for (int ox0 = 0; ox0 < a.ow; ox0 += 4) {
        float g[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) g[j] = (cok && ox0 + j < a.ow) ? __bfloat162float(dyrow[(long long)(ox0 + j) * a.lddy]) : 0.f;
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci)
#pragma unroll
          for (int kz = 0; kz < 3; ++kz)
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
              const float* xr = sx + ((ci * 3 + kz) * 10 + warp + ky) * Wa + ox0;
              float xv[6];
#pragma unroll
              for (int j = 0; j < 6; ++j) xv[j] = xr[j];
#pragma unroll
              for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                  acc[ci * 27 + (kz * 3 + ky) * 3 + kx] = fmaf(g[j], xv[j + kx], acc[ci * 27 + (kz * 3 + ky) * 3 + kx]);
            }
      }
    }
  }
  float* red = sx;  // [8][27][32]
#pragma unroll
  for (int ci = 0; ci < CIN; ++ci) {
    __syncthreads();
#pragma unroll
    for (int t = 0; t < 27; ++t) red[(warp * 27 + t) * 32 + lane] = acc[ci * 27 + t];
    __syncthreads();
    for (int i = threadIdx.x; i < 27 * 32; i += 256) {
      const int t = i / 32, l = i % 32;
      float sum = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) sum += red[(w * 27 + t) * 32 + l];
      if (blockIdx.y * 32 + l < a.cout)
        a.ws[(((long long)ci * gridDim.x + blockIdx.x) * kWgAcc + t) * a.cout + blockIdx.y * 32 + l] = sum;
    }
  }
}

template <int CIN>
static int launch_smallcin_wgrad_k3(const SmallCinWgradArgs& a, cudaStream_t stream) {
  const size_t smem = std::max<size_t>((size_t)CIN * 30 * (a.wd + 6) * sizeof(float), (size_t)8 * 27 * 32 * sizeof(float));
  if (smem > 200 * 1024) return REHR_UNSUPPORTED;
  static size_t attr_smem = 0;
  if (smem > 48 * 1024 && smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(smallcin_wgrad_k3_kernel<CIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      g_last_cuda_error = (int)e;
      return REHR_CUDA_ERROR;
    }
    attr_smem = smem;
  }
  dim3 grid(kWgBlocks, (a.cout + 31) / 32);
  smallcin_wgrad_k3_kernel<CIN><<<grid, 256, smem, stream>>>(a);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

// General row-staged variant for larger in-plane kernels / strides (the FLAVR stem k(3,7,7) s(1,2,2), resnet_3D.py:42-50):
// one launch covers all (ci, kz) pairs through blockIdx.z, each CTA stages the (7*SH + KH) input rows that 8 output rows need
// for that (ci, kz) into shared memory, lane = output channel, KH*KW register accumulators per thread, 4 output voxels per
// inner iteration.  Partials: ws[block][(ci*KD + kz)*KH*KW + ky*KW + kx][cout].
template <int KH, int KW, int SH, int SW>
__global__ void __launch_bounds__(256) smallcin_wgrad_rows_kernel(const SmallCinWgradArgs a) {
  extern __shared__ float sx[];  // [7*SH + KH][Wa], then reused as red[8][KH*KW][32]
  constexpr int T2 = KH * KW;
  constexpr int ROWS = 7 * SH + KH;
  constexpr int SPAN = 3 * SW + KW;  // input columns touched by 4 consecutive output voxels
  const int Wa = a.wd + 2 * a.pw + SPAN + 4;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int co = blockIdx.y * 32 + lane;
  const bool cok = co < a.cout;
  const int ci = blockIdx.z / a.kd, kz = blockIdx.z % a.kd;
  float acc[T2];
#pragma unroll
  for (int i = 0; i < T2; ++i) acc[i] = 0.f;
  const int ytiles = (a.oh + 7) / 8;
  const long long tiles = (long long)a.n * a.od * ytiles;
  const long long in_plane = (long long)a.h * a.wd, in_vol = in_plane * a.d;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int yt = (int)(tile % ytiles);
    long long r = tile / ytiles;
    const int oz = (int)(r % a.od);
    const int nn = (int)(r / a.od);
    const int oy0 = yt * 8;
    const int iz = oz * a.sd + kz - a.pd;
    if (iz < 0 || iz >= a.d) continue;  // whole (tile, kz) reads padding: contributes nothing (uniform across the CTA)
    __syncthreads();
    const float* xp = a.x + ((long long)nn * a.cin + ci) * in_vol + (long long)iz * in_plane;
    for (int i = threadIdx.x; i < ROWS * Wa; i += 256) {
      const int xx = i % Wa, rr = i / Wa;
      const int iy = oy0 * SH + rr - a.ph, ix = xx - a.pw;
      sx[i] = (iy >= 0 && iy < a.h && ix >= 0 && ix < a.wd) ? __ldg(xp + (long long)iy * a.wd + ix) : 0.f;
    }
    __syncthreads();
    const int oy = oy0 + warp;
    if (oy < a.oh) {
      const __nv_bfloat16* dyrow = a.dy + ((((long long)nn * a.od + oz) * a.oh + oy) * a.ow) * a.lddy + co;
      for (int ox0 = 0; ox0 < a.ow; ox0 += 4) {
        float g[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) g[j] = (cok && ox0 + j < a.ow) ? __bfloat162float(dyrow[(long long)(ox0 + j) * a.lddy]) : 0.f;
#pragma unroll
        for (int ky = 0; ky < KH; ++ky) {
          const float* xr = sx + (warp * SH + ky) * Wa + ox0 * SW;
          float xv[SPAN];
#pragma unroll
          for (int j = 0; j < SPAN; ++j) xv[j] = xr[j];
#pragma unroll
          for (int kx = 0; kx < KW; ++kx)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[ky * KW + kx] = fmaf(g[j], xv[j * SW + kx], acc[ky * KW + kx]);
        }
      }
    }
  }
  float* red = sx;  // [8][T2][32]
  __syncthreads();
#pragma unroll
  for (int t = 0; t < T2; ++t) red[(warp * T2 + t) * 32 + lane] = acc[t];
  __syncthreads();
  const int KT = a.cin * a.kd * T2;
  for (int i = threadIdx.x; i < T2 * 32; i += 256) {
    const int t = i / 32, l = i % 32;
    float sum = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) sum += red[(w * T2 + t) * 32 + l];
    if (blockIdx.y * 32 + l < a.cout)
      a.ws[((long long)blockIdx.x * KT + (long long)blockIdx.z * T2 + t) * a.cout + blockIdx.y * 32 + l] = sum;
  }
}

// ws[block][k][cout] -> dw[co][k]  (k = (ci*KD + kz)*KH*KW + t2 is exactly PyTorch's [ci][kz][ky][kx] order)
__global__ void smallcin_wgrad_rows_reduce_kernel(const float* ws, int blocks, int KT, int cout, float* dw, int accumulate) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= KT * cout) return;
  const int co = i % cout, k = i / cout;
  float s = 0.f;
  for (int b = 0; b < blocks; ++b) s += ws[((long long)b * KT + k) * cout + co];
  float* d = dw + (long long)co * KT + k;
  *d = accumulate ? *d + s : s;
}

static constexpr int kWgRowsBlocks = 296;  // 2 x 148 CTAs per (channel block, (ci, kz)) slice

__global__ void smallcin_wgrad_reduce_kernel(const float* ws, int blocks, int passes, int KT, int cout, float* dw,
                                             int accumulate) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= KT * cout) return;
  const int co = i % cout, k = i / cout;
  const int pass = k / kWgAcc, kk = k % kWgAcc;
  (void)passes;
  float s = 0.f;
  for (int b = 0; b < blocks; ++b) s += ws[(((long long)pass * blocks + b) * kWgAcc + kk) * cout + co];
  float* d = dw + (long long)co * KT + k;
  *d = accumulate ? *d + s : s;
}

// Input gradient (gather form): dx[n][ci][i] = sum_{co,t : (i+p-t) % s == 0} dy[(i+p-t)/s, co] * w[co][ci][t]
struct SmallCinDgradArgs {
  const __nv_bfloat16* dy;
  long long lddy;
  const float* w;
  float* dx;
  int n, cin, d, h, wd, od, oh, ow, cout;
  int kd, kh, kw, sd, sh, sw, pd, ph, pw;
};

__global__ void __launch_bounds__(256) smallcin_dgrad_kernel(const SmallCinDgradArgs a) {
  const int T = a.kd * a.kh * a.kw;
  const long long ivox = (long long)a.n * a.d * a.h * a.wd;
  for (long long it = blockIdx.x * (long long)blockDim.x + threadIdx.x; it < ivox * a.cin; it += (long long)gridDim.x * blockDim.x) {
    const int ci = (int)(it / ivox);
    long long v = it % ivox;
    const int ix = (int)(v % a.wd);
    long long r = v / a.wd;
    const int iy = (int)(r % a.h);
    r /= a.h;
    const int iz = (int)(r % a.d);
    const int nn = (int)(r / a.d);
    float acc = 0.f;
    for (int kz = 0; kz < a.kd; ++kz) {
      const int ez = iz + a.pd - kz;
      if (ez < 0 || ez % a.sd != 0 || ez / a.sd >= a.od) continue;
      for (int ky = 0; ky < a.kh; ++ky) {
        const int ey = iy + a.ph - ky;
        if (ey < 0 || ey % a.sh != 0 || ey / a.sh >= a.oh) continue;
        for (int kx = 0; kx < a.kw; ++kx) {
          const int ex = ix + a.pw - kx;
          if (ex < 0 || ex % a.sw != 0 || ex / a.sw >= a.ow) continue;
          const long long o = (((long long)nn * a.od + ez / a.sd) * a.oh + ey / a.sh) * a.ow + ex / a.sw;
          const int t = (kz * a.kh + ky) * a.kw + kx;
          const __nv_bfloat16* g = a.dy + o * a.lddy;
          for (int co = 0; co < a.cout; ++co) acc = fmaf(__bfloat162float(g[co]), __ldg(a.w + ((long long)co * a.cin + ci) * T + t), acc);
        }
      }
    }
    a.dx[((long long)nn * a.cin + ci) * ((long long)a.d * a.h * a.wd) + ((long long)iz * a.h + iy) * a.wd + ix] = acc;
  }
}

}  // namespace rehr

using namespace rehr;

namespace {
inline int conv_out(int in, int k, int s, int p) { return (in + 2 * p - k) / s + 1; }
bool shapes_ok(const rehr_conv_desc* d, int n, int cin, int D, int H, int W, const rehr_tensor* y) {
  if (!d || !y || !y->ptr || n <= 0 || cin <= 0 || cin > kScMaxCin) return false;
  if (y->n != n) return false;
  return y->d == conv_out(D, d->kd, d->sd, d->pd) && y->h == conv_out(H, d->kh, d->sh, d->ph) &&
         y->w == conv_out(W, d->kw, d->sw, d->pw);
}
}  // namespace

extern "C" {

int rehr_instnorm_stats(const rehr_tensor* x, float* partial, rehr_stream stream);

int rehr_conv3d_smallcin_fwd(const rehr_conv_desc* desc, const float* x_ncdhw, int n, int cin, int d, int h, int w,
                             const float* weight, const float* bias, const rehr_tensor* y, int act, float slope,
                             float* stats, rehr_stream stream) {
  if (!shapes_ok(desc, n, cin, d, h, w, y) || !x_ncdhw || !weight) return REHR_BAD_SHAPE;
  if (y->ld % 8 != 0 || (reinterpret_cast<uintptr_t>(y->ptr) & 15) != 0) return REHR_BAD_ALIGNMENT;
  if (y->c % 4 != 0) return REHR_UNSUPPORTED;
  const int T = desc->kd * desc->kh * desc->kw;
  const size_t smem = (size_t)cin * T * y->c * sizeof(float);
  if (smem > 200 * 1024) return REHR_UNSUPPORTED;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(smallcin_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      g_last_cuda_error = (int)e;
      return REHR_CUDA_ERROR;
    }
  }
  SmallCinArgs a;
  a.x = x_ncdhw;
  a.w = weight;
  a.bias = bias;
  a.y = reinterpret_cast<__nv_bfloat16*>(y->ptr);
  a.ldy = y->ld;
  a.n = n; a.cin = cin; a.d = d; a.h = h; a.wd = w;
  a.od = y->d; a.oh = y->h; a.ow = y->w; a.cout = y->c;
  a.kd = desc->kd; a.kh = desc->kh; a.kw = desc->kw;
  a.sd = desc->sd; a.sh = desc->sh; a.sw = desc->sw;
  a.pd = desc->pd; a.ph = desc->ph; a.pw = desc->pw;
  a.act = act;
  a.slope = slope;
  a.y_f16 = y->dtype == REHR_F16;
  a.range = range_target(a.y_f16);
  const bool k3 = desc->kd == 3 && desc->kh == 3 && desc->kw == 3 && desc->sd == 1 && desc->sh == 1 && desc->sw == 1 &&
                  desc->pd == 1 && desc->ph == 1 && desc->pw == 1;
  // planar stem of anisotropic plans: k = (1,3,3), stride 1, pad (0,1,1)
  const bool k133 = desc->kd == 1 && desc->kh == 3 && desc->kw == 3 && desc->sd == 1 && desc->sh == 1 && desc->sw == 1 &&
                    desc->pd == 0 && desc->ph == 1 && desc->pw == 1;
  int rc = REHR_UNSUPPORTED;
  if ((k3 || k133) && stem_mma_supported(cin, y->c, w) && y->ld % 8 == 0) {
    rc = launch_stem_fwd_mma(x_ncdhw, weight, bias, a.y, a.ldy, a.y_f16, n, d, h, w, act, slope, k133 ? 1 : 0, (cudaStream_t)stream);
    if (rc != REHR_OK && rc != REHR_UNSUPPORTED) return rc;
  }
  if (rc == REHR_UNSUPPORTED && k3 && y->c == 32 && cin <= 2) {
    rc = cin == 1 ? launch_smallcin_fwd_k3c32<1>(a, (cudaStream_t)stream) : launch_smallcin_fwd_k3c32<2>(a, (cudaStream_t)stream);
    if (rc != REHR_OK && rc != REHR_UNSUPPORTED) return rc;
  }
  if (rc == REHR_UNSUPPORTED) {
    const long long items = (long long)n * y->d * y->h * y->w * ((y->c + kScCoutPerThread - 1) / kScCoutPerThread);
    const int blocks = (int)std::max<long long>(1, std::min<long long>((items + 255) / 256, (long long)sm_count() * 8));
    smallcin_fwd_kernel<<<blocks, 256, smem, (cudaStream_t)stream>>>(a);
    REHR_CHECK_LAUNCH();
  }
  if (stats) {
    if (act != REHR_ACT_NONE) return REHR_UNSUPPORTED;  // statistics are defined on the pre-activation output
    return rehr_instnorm_stats(y, stats, stream);
  }
  return REHR_OK;
}

static bool smallcin_rows_variant(const rehr_conv_desc* d) {
  return d->kh == 7 && d->kw == 7 && d->sh == 2 && d->sw == 2;
}

size_t rehr_conv3d_smallcin_wgrad_workspace(const rehr_conv_desc* desc, int cin, const rehr_tensor* dy) {
  if (!desc || !dy || cin <= 0 || cin > kScMaxCin) return 0;
  const int KT = cin * desc->kd * desc->kh * desc->kw;
  const int passes = (KT + kWgAcc - 1) / kWgAcc;
  const size_t generic = (size_t)passes * kWgBlocks * kWgAcc * dy->c * sizeof(float);
  const size_t rows = smallcin_rows_variant(desc) ? (size_t)kWgRowsBlocks * KT * dy->c * sizeof(float) : 0;
  return std::max(generic, rows);
}

int rehr_conv3d_smallcin_wgrad(const rehr_conv_desc* desc, const float* x_ncdhw, int n, int cin, int d, int h, int w,
                               const rehr_tensor* dy, float* dw, int accumulate, void* ws, size_t ws_bytes,
                               rehr_stream stream) {
  if (!shapes_ok(desc, n, cin, d, h, w, dy) || !x_ncdhw || !dw) return REHR_BAD_SHAPE;
  const size_t need = rehr_conv3d_smallcin_wgrad_workspace(desc, cin, dy);
  if (!ws || ws_bytes < need) return REHR_WORKSPACE;
  const int KT = cin * desc->kd * desc->kh * desc->kw;
  const int passes = (KT + kWgAcc - 1) / kWgAcc;
  SmallCinWgradArgs a;
  a.x = x_ncdhw;
  a.dy = reinterpret_cast<const __nv_bfloat16*>(dy->ptr);
  a.lddy = dy->ld;
  a.ws = reinterpret_cast<float*>(ws);
  a.n = n; a.cin = cin; a.d = d; a.h = h; a.wd = w;
  a.od = dy->d; a.oh = dy->h; a.ow = dy->w; a.cout = dy->c;
  a.kd = desc->kd; a.kh = desc->kh; a.kw = desc->kw;
  a.sd = desc->sd; a.sh = desc->sh; a.sw = desc->sw;
  a.pd = desc->pd; a.ph = desc->ph; a.pw = desc->pw;
  const bool k3 = desc->kd == 3 && desc->kh == 3 && desc->kw == 3 && desc->sd == 1 && desc->sh == 1 && desc->sw == 1 &&
                  desc->pd == 1 && desc->ph == 1 && desc->pw == 1;
  const bool k133 = desc->kd == 1 && desc->kh == 3 && desc->kw == 3 && desc->sd == 1 && desc->sh == 1 && desc->sw == 1 &&
                    desc->pd == 0 && desc->ph == 1 && desc->pw == 1;
  int rc = REHR_UNSUPPORTED;
  if ((k3 || k133) && stem_mma_supported(cin, dy->c, w) && dy->ld % 8 == 0 && ws_bytes >= stem_mma_wgrad_workspace())
    return launch_stem_wgrad_mma(x_ncdhw, a.dy, a.lddy, n, d, h, w, dw, accumulate, a.ws, k133 ? 1 : 0, (cudaStream_t)stream);
  if (k3) {
    switch (cin) {
      case 1: rc = launch_smallcin_wgrad_k3<1>(a, (cudaStream_t)stream); break;
      case 2: rc = launch_smallcin_wgrad_k3<2>(a, (cudaStream_t)stream); break;
      case 3: rc = launch_smallcin_wgrad_k3<3>(a, (cudaStream_t)stream); break;
      case 4: rc = launch_smallcin_wgrad_k3<4>(a, (cudaStream_t)stream); break;
      default: break;
    }
    if (rc != REHR_OK && rc != REHR_UNSUPPORTED) return rc;
  }
  if (rc == REHR_UNSUPPORTED && smallcin_rows_variant(desc)) {
    constexpr int ROWS = 7 * 2 + 7, SPAN = 3 * 2 + 7;
    const int Wa = w + 2 * desc->pw + SPAN + 4;
    const size_t smem = std::max<size_t>((size_t)ROWS * Wa * sizeof(float), (size_t)8 * 49 * 32 * sizeof(float));
    if (smem <= 200 * 1024) {
      static size_t attr_smem = 0;
      if (smem > 48 * 1024 && smem > attr_smem) {
        cudaError_t e = cudaFuncSetAttribute(smallcin_wgrad_rows_kernel<7, 7, 2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) {
          g_last_cuda_error = (int)e;
          return REHR_CUDA_ERROR;
        }
        attr_smem = smem;
      }
      dim3 grid(kWgRowsBlocks, (dy->c + 31) / 32, cin * desc->kd);
      smallcin_wgrad_rows_kernel<7, 7, 2, 2><<<grid, 256, smem, (cudaStream_t)stream>>>(a);
      REHR_CHECK_LAUNCH();
      const int total = KT * dy->c;
      smallcin_wgrad_rows_reduce_kernel<<<(total + 127) / 128, 128, 0, (cudaStream_t)stream>>>(a.ws, kWgRowsBlocks, KT, dy->c, dw,
                                                                                             accumulate);
      REHR_CHECK_LAUNCH();
      return REHR_OK;
    }
  }
  if (rc == REHR_UNSUPPORTED) {
    dim3 grid(kWgBlocks, passes);
    smallcin_wgrad_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    REHR_CHECK_LAUNCH();
  }
  const int total = KT * dy->c;
  smallcin_wgrad_reduce_kernel<<<(total + 127) / 128, 128, 0, (cudaStream_t)stream>>>(a.ws, kWgBlocks, passes, KT, dy->c, dw,
                                                                                     accumulate);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_conv3d_smallcin_dgrad(const rehr_conv_desc* desc, const rehr_tensor* dy, const float* weight, float* dx_ncdhw,
                               int n, int cin, int d, int h, int w, rehr_stream stream) {
  if (!shapes_ok(desc, n, cin, d, h, w, dy) || !weight || !dx_ncdhw) return REHR_BAD_SHAPE;
  SmallCinDgradArgs a;
  a.dy = reinterpret_cast<const __nv_bfloat16*>(dy->ptr);
  a.lddy = dy->ld;
  a.w = weight;
  a.dx = dx_ncdhw;
  a.n = n; a.cin = cin; a.d = d; a.h = h; a.wd = w;
  a.od = dy->d; a.oh = dy->h; a.ow = dy->w; a.cout = dy->c;
  a.kd = desc->kd; a.kh = desc->kh; a.kw = desc->kw;
  a.sd = desc->sd; a.sh = desc->sh; a.sw = desc->sw;
  a.pd = desc->pd; a.ph = desc->ph; a.pw = desc->pw;
  const long long items = (long long)n * cin * d * h * w;
  const int blocks = (int)std::max<long long>(1, std::min<long long>((items + 255) / 256, (long long)sm_count() * 8));
  smallcin_dgrad_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(a);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

}  // extern "C"
