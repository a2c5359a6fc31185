// HBM-bound kernels of the hot path: InstanceNorm(+LeakyReLU) forward/backward, the 1x1x1 segmentation head,
// layout adapters, depth-linear upsampling, SE-gate tail, sliding-window Gaussian blend, blur stencil, rot90,
// FBA spectral combine.  All are vectorised (16 B per thread access where the layout allows), coalesced and
// sized as a multiple of the SM count; reductions are shuffle / shared-memory trees with deterministic
// per-block partials (no float atomics on global memory).
#include "engine.h"
#include "bspline.cuh"
#include "ptx.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cstdlib>

namespace rehr {

static inline int grid_for(long long work_items, int threads, int waves = 8) {
  long long b = (work_items + threads - 1) / threads;
  long long cap = (long long)sm_count() * waves;
  return (int)std::max<long long>(1, std::min<long long>(b, cap));
}

__device__ __forceinline__ void bf16x8_to_float(const uint4& u, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 float_to_bf16x8(const float (&f)[8]) {
  uint4 u;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return u;
}

// 16-bit payloads of either storage format (rehr_tensor.dtype): fp16 != 0 selects fp16, else bf16
__device__ __forceinline__ void x16x8_to_float(const uint4& u, float (&f)[8], int fp16) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = unpack16x2(w[i], fp16);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 float_to_x16x8(const float (&f)[8], int fp16) {
  return make_uint4(pack16x2(f[0], f[1], fp16), pack16x2(f[2], f[3], fp16), pack16x2(f[4], f[5], fp16), pack16x2(f[6], f[7], fp16));
}

static bool bf16_tensor_ok(const rehr_tensor* t) {
  return t && t->ptr && t->c % 8 == 0 && t->ld % 8 == 0 && (reinterpret_cast<uintptr_t>(t->ptr) & 15) == 0;
}
static inline long long voxels_per_sample(const rehr_tensor* t) { return (long long)t->d * t->h * t->w; }

// =================================================================================================
// InstanceNorm statistics (stand-alone; the conv epilogue normally produces these)
// =================================================================================================
static constexpr int kStatThreads = 256;
static constexpr int kStatMaxVoxPerBlock = 2048;

// Voxels per reduction block: as many as 2048 (full-resolution tensors: ~1000+ blocks), but never so many that a
// small deep-layer tensor is reduced by a handful of blocks (aim for >= 2 blocks per SM across the batch).
static int stat_vox_per_block(const rehr_tensor* x) {
  const long long V = (long long)x->d * x->h * x->w;
  const int groups = std::max(1, x->c / 8);
  const int lanes = std::max(1, kStatThreads / groups);
  const long long want_tiles = std::max<long long>(1, (2LL * sm_count() + x->n - 1) / std::max(1, x->n));
  long long vpb = (V + want_tiles - 1) / want_tiles;
  vpb = std::max<long long>(vpb, (long long)lanes * 4);
  vpb = std::min<long long>(vpb, kStatMaxVoxPerBlock);
  vpb = (vpb + lanes - 1) / lanes * lanes;
  return (int)vpb;
}

// Block = (tile, n).  Thread = (voxel lane, channel group of 8).  Per-thread accumulation, then a
// shared-memory tree over voxel lanes.  `mode` 0: (sum x, sum x^2); 1: InstanceNorm backward sums.
struct StatArgs {
  const __nv_bfloat16* y;
  const __nv_bfloat16* da1;
  const __nv_bfloat16* da2;
  long long ld_y, ld_a1, ld_a2;
  const float *mean, *rstd, *gamma, *beta;
  float slope;
  float* partial;
  long long V;
  int C, tiles, vpb;
  int y_f16;  // storage format of y (the gradients da1 / da2 are always bf16)
};

template <int MODE>
__global__ void __launch_bounds__(kStatThreads) in_reduce_kernel(const StatArgs a) {
  extern __shared__ float sh[];  // [lanes][C][2]
  const int n = blockIdx.y, tile = blockIdx.x;
  const int groups = a.C / 8;
  const int lanes = kStatThreads / groups;  // voxel lanes per pass (>=1)
  const int g = threadIdx.x % groups, vl = threadIdx.x / groups;
  const long long v0 = (long long)tile * a.vpb;
  const long long v1 = min(a.V, v0 + a.vpb);
  float s1[8], s2[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s1[i] = s2[i] = 0.f;
  float sc[8], sf[8], mu[8], rs[8];
  if (MODE == 1) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = g * 8 + i;
      mu[i] = a.mean[n * a.C + c];
      rs[i] = a.rstd[n * a.C + c];
      sc[i] = a.gamma ? a.gamma[c] : 1.f;
      sf[i] = a.beta ? a.beta[c] : 0.f;
    }
  }
  if (vl < lanes) {
    constexpr int U = 4;  // voxels in flight per thread: all loads of a batch are issued before any arithmetic
    for (long long vb = v0 + vl; vb < v1; vb += (long long)lanes * U) {
      uint4 yv[U], dv[U], ev[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long v = vb + (long long)u * lanes;
        if (v < v1) {
          const long long vox = (long long)n * a.V + v;
          yv[u] = *reinterpret_cast<const uint4*>(a.y + vox * a.ld_y + g * 8);
          if (MODE == 1) {
            dv[u] = *reinterpret_cast<const uint4*>(a.da1 + vox * a.ld_a1 + g * 8);
            if (a.da2) ev[u] = *reinterpret_cast<const uint4*>(a.da2 + vox * a.ld_a2 + g * 8);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long v = vb + (long long)u * lanes;
        if (v >= v1) break;
        float y[8];
        x16x8_to_float(yv[u], y, a.y_f16);
        if (MODE == 0) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            s1[i] += y[i];
            s2[i] += y[i] * y[i];
          }
        } else {
          float d[8];
          bf16x8_to_float(dv[u], d);
          if (a.da2) {
            float d2[8];
            bf16x8_to_float(ev[u], d2);
#pragma unroll
            for (int i = 0; i < 8; ++i) d[i] += d2[i];
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float xh = (y[i] - mu[i]) * rs[i];
            const float z = sc[i] * xh + sf[i];
            const float gi = z > 0.f ? d[i] : d[i] * a.slope;
            s1[i] += gi;
            s2[i] += gi * xh;
          }
        }
      }
    }
  }
  if (vl < lanes) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      sh[(vl * a.C + g * 8 + i) * 2] = s1[i];
      sh[(vl * a.C + g * 8 + i) * 2 + 1] = s2[i];
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < a.C; c += kStatThreads) {
    float t1 = 0.f, t2 = 0.f;
    for (int l = 0; l < lanes; ++l) {
      t1 += sh[(l * a.C + c) * 2];
      t2 += sh[(l * a.C + c) * 2 + 1];
    }
    float* dst = a.partial + (((long long)n * a.tiles + tile) * a.C + c) * 2;
    dst[0] = t1;
    dst[1] = t2;
  }
}

static int stat_tiles(const rehr_tensor* x) {
  const long long V = voxels_per_sample(x);
  const int vpb = stat_vox_per_block(x);
  return (int)((V + vpb - 1) / vpb);
}

template <int MODE>
static int launch_in_reduce(const StatArgs& a, int N, cudaStream_t st) {
  const int groups = a.C / 8;
  if (groups > kStatThreads) return REHR_UNSUPPORTED;
  const int lanes = kStatThreads / groups;
  const size_t smem = (size_t)lanes * a.C * 2 * sizeof(float);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(in_reduce_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      g_last_cuda_error = (int)e;
      return REHR_CUDA_ERROR;
    }
  }
  dim3 grid(a.tiles, N);
  in_reduce_kernel<MODE><<<grid, kStatThreads, smem, st>>>(a);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

// partial [n][tiles][c][2] -> mean, rstd.  Block = (32 channels) x (32 tile lanes); grid = (C/32 ceil, N).  The tile
// lanes stride through the partial list (coalesced 256 B rows), accumulate in double and meet in a shared-memory tree,
// so a 1024-tile list costs ~32 dependent-free loads per thread instead of 1024 serial ones.
static constexpr int kFinLanes = 32;

// CPB = channels per block (32, or 8 for long partial lists: four times as many blocks and tile lanes -- the stage-entry convs
// leave 2048 partials per sample, which 4 blocks of 32 lanes took 25 us to walk)
template <int CPB>
__global__ void __launch_bounds__(32 * kFinLanes) in_finalize_kernel(const float* partial, int N, int tiles, int C,
                                                                      double inv_count, float eps, float* mean, float* rstd) {
  constexpr int kLanes = 32 * kFinLanes / CPB;
  __shared__ double sh1[kLanes][CPB + 1], sh2[kLanes][CPB + 1];
  const int cl = threadIdx.x % CPB, tl = threadIdx.x / CPB;
  const int n = blockIdx.y, c = blockIdx.x * CPB + cl;
  double s1 = 0.0, s2 = 0.0;
  if (c < C) {
    const float2* p = reinterpret_cast<const float2*>(partial) + (long long)n * tiles * C + c;
#pragma unroll 8
    for (int t = tl; t < tiles; t += kLanes) {
      const float2 v = p[(long long)t * C];
      s1 += (double)v.x;
      s2 += (double)v.y;
    }
  }
  sh1[tl][cl] = s1;
  sh2[tl][cl] = s2;
  __syncthreads();
  if (tl == 0 && c < C) {
    double a = 0.0, b = 0.0;
#pragma unroll 8
    for (int l = 0; l < kLanes; ++l) {
      a += sh1[l][cl];
      b += sh2[l][cl];
    }
    const double m = a * inv_count;
    double var = b * inv_count - m * m;
    if (var < 0.0) var = 0.0;
    const float rs = (float)(1.0 / sqrt(var + (double)eps));
    mean[n * C + c] = (float)m;
    rstd[n * C + c] = rs;
  }
}

// partial [n][tiles][c][2] -> sums [n][c][2]; dgamma[c] = sum_n S2, dbeta[c] = sum_n S1.  Same thread layout; grid = C/32.
__global__ void __launch_bounds__(32 * kFinLanes) in_bwd_finalize_kernel(const float* partial, int N, int tiles, int C,
                                                                          float* sums, float* dgamma, float* dbeta,
                                                                          int accumulate) {
  __shared__ double sh1[kFinLanes][33], sh2[kFinLanes][33];
  const int cl = threadIdx.x & 31, tl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  double g = 0.0, b = 0.0;
  // two samples per pass: their partial lists are independent, so twice as many loads are in flight per round trip
  for (int n0 = 0; n0 < N; n0 += 2) {
    const bool two = n0 + 1 < N;
    double s1a = 0.0, s2a = 0.0, s1b = 0.0, s2b = 0.0;
    if (c < C) {
      const float2* pa = reinterpret_cast<const float2*>(partial) + (long long)n0 * tiles * C + c;
      const float2* pb = pa + (two ? (long long)tiles * C : 0);
#pragma unroll 8
      for (int t = tl; t < tiles; t += kFinLanes) {
        const float2 va = pa[(long long)t * C];
        const float2 vb = pb[(long long)t * C];
        s1a += (double)va.x;
        s2a += (double)va.y;
        s1b += (double)vb.x;
        s2b += (double)vb.y;
      }
    }
    for (int k = 0; k < (two ? 2 : 1); ++k) {
      __syncthreads();
      sh1[tl][cl] = k == 0 ? s1a : s1b;
      sh2[tl][cl] = k == 0 ? s2a : s2b;
      __syncthreads();
      if (tl == 0 && c < C) {
        double a1 = 0.0, a2 = 0.0;
#pragma unroll
        for (int l = 0; l < kFinLanes; ++l) {
          a1 += sh1[l][cl];
          a2 += sh2[l][cl];
        }
        const int n = n0 + k;
        sums[((long long)n * C + c) * 2] = (float)a1;
        sums[((long long)n * C + c) * 2 + 1] = (float)a2;
        b += a1;
        g += a2;
      }
    }
  }
  if (tl == 0 && c < C) {
    if (dgamma) dgamma[c] = accumulate ? dgamma[c] + (float)g : (float)g;
    if (dbeta) dbeta[c] = accumulate ? dbeta[c] + (float)b : (float)b;
  }
}

struct ApplyArgs {
  const __nv_bfloat16* y;
  const __nv_bfloat16* da1;
  const __nv_bfloat16* da2;
  __nv_bfloat16* out;
  long long ld_y, ld_a1, ld_a2, ld_o;
  const float *mean, *rstd, *gamma, *beta, *sums;
  float slope;
  long long V;
  int C;
  int y_f16, out_f16;    // storage formats of y and out (da1 / da2 are always bf16)
  __nv_bfloat16* out2;   // MODE 0 only: optional second copy of the activation in the other 16-bit format (may be null)
  long long ld_o2;
  int out2_f16;
  RangeSlot* range;      // MODE 0 only: fp16 saturation record of out (rehr_range_sink), null = not checked
};

// MODE 0: a = lrelu(gamma*xhat + beta).  MODE 1: dy = gamma*rstd*(g - S1/V - xhat*S2/V).
// RC (MODE 0): the fp16 saturation check of a (a.range != null) is compiled in; the unchecked instantiation has no trace of it.
template <int MODE, bool RC = false>
__global__ void __launch_bounds__(256, MODE == 1 ? 4 : 1) in_apply_kernel(const ApplyArgs a) {
  extern __shared__ float sh[];  // MODE0: scale, shift ; MODE1: mean, rstd, gamma, beta, m1, m2
  const int n = blockIdx.y;
  const int C = a.C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float mu = a.mean[n * C + c], rs = a.rstd[n * C + c];
    const float ga = a.gamma ? a.gamma[c] : 1.f, be = a.beta ? a.beta[c] : 0.f;
    if (MODE == 0) {
      sh[c] = ga * rs;
      sh[C + c] = be - mu * ga * rs;
    } else {
      sh[c] = mu;
      sh[C + c] = rs;
      sh[2 * C + c] = ga;
      sh[3 * C + c] = be;
      sh[4 * C + c] = a.sums[((long long)n * C + c) * 2] / (float)a.V;
      sh[5 * C + c] = a.sums[((long long)n * C + c) * 2 + 1] / (float)a.V;
    }
  }
  __syncthreads();
  const int groups = C / 8;
  const long long items = a.V * groups;
  const long long stride = (long long)gridDim.x * blockDim.x;
  constexpr int U = 2;  // items in flight per thread: both batches of loads are issued before the arithmetic
  for (long long it0 = blockIdx.x * (long long)blockDim.x + threadIdx.x; it0 < items; it0 += stride * U) {
    uint4 yv[U], dv[U], ev[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long it = it0 + u * stride;
      if (it < items) {
        const int g = (int)(it % groups);
        const long long vox = (long long)n * a.V + it / groups;
        yv[u] = __ldcs(reinterpret_cast<const uint4*>(a.y + vox * a.ld_y + g * 8));
        if (MODE == 1) {
          dv[u] = __ldcs(reinterpret_cast<const uint4*>(a.da1 + vox * a.ld_a1 + g * 8));
          if (a.da2) ev[u] = __ldcs(reinterpret_cast<const uint4*>(a.da2 + vox * a.ld_a2 + g * 8));
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long it = it0 + u * stride;
      if (it >= items) break;
      const int g = (int)(it % groups);
      const long long vox = (long long)n * a.V + it / groups;
      float y[8], o[8];
      x16x8_to_float(yv[u], y, a.y_f16);
      if (MODE == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float z = y[i] * sh[g * 8 + i] + sh[C + g * 8 + i];
          o[i] = z > 0.f ? z : z * a.slope;
        }
      } else {
        float d[8];
        bf16x8_to_float(dv[u], d);
        if (a.da2) {
          float d2[8];
          bf16x8_to_float(ev[u], d2);
#pragma unroll
          for (int i = 0; i < 8; ++i) d[i] += d2[i];
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int c = g * 8 + i;
          const float xh = (y[i] - sh[c]) * sh[C + c];
          const float z = sh[2 * C + c] * xh + sh[3 * C + c];
          const float gi = z > 0.f ? d[i] : d[i] * a.slope;
          o[i] = sh[2 * C + c] * sh[C + c] * (gi - sh[4 * C + c] - xh * sh[5 * C + c]);
        }
      }
      if constexpr (RC) range_check<8>(a.range, o);
      *reinterpret_cast<uint4*>(a.out + vox * a.ld_o + g * 8) = float_to_x16x8(o, a.out_f16);
      if (MODE == 0 && a.out2 != nullptr) *reinterpret_cast<uint4*>(a.out2 + vox * a.ld_o2 + g * 8) = float_to_x16x8(o, a.out2_f16);
    }
  }
}

template <int MODE>
static int launch_in_apply(const ApplyArgs& a, int N, cudaStream_t st) {
  const size_t smem = (size_t)(MODE == 0 ? 2 : 6) * a.C * sizeof(float);
  const long long items = a.V * (a.C / 8);
  int gx = grid_for(items, 256, 8);
  gx = std::max(1, gx / std::max(1, N));
  dim3 grid(gx, N);
  bool checked = false;
  if constexpr (MODE == 0) {
    if (a.range != nullptr) {
      in_apply_kernel<0, true><<<grid, 256, smem, st>>>(a);
      checked = true;
    }
  }
  if (!checked) in_apply_kernel<MODE, false><<<grid, 256, smem, st>>>(a);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

// =================================================================================================
// 1x1x1 conv to a few channels (segmentation head), NDHWC bf16 -> NCDHW f32
// =================================================================================================
static constexpr int kPwCoutLimit = 8;
static constexpr int kPwMaxCin = 128;

// kPwMaxCout: compile-time bound on cout (2 / 4 / 8) -- keeps the accumulators in a few registers.  CIN > 0: compile-time
// channel count (all 16-byte loads of a voxel are issued before the arithmetic); CIN = 0: run-time cin.  grid = (blocks, N):
// the sample index comes from blockIdx.y, so the voxel loop carries no 64-bit division.
template <int kPwMaxCout, int CIN>
__global__ void __launch_bounds__(256) pointwise_fwd_kernel(const __nv_bfloat16* x, long long ld, const float* w,
                                                            const float* bias, float* y, long long V, int cin_rt, int cout,
                                                            int x_f16) {
  const int cin = CIN > 0 ? CIN : cin_rt;
  __shared__ float sw[kPwMaxCout * kPwMaxCin + kPwMaxCout];
  for (int i = threadIdx.x; i < cout * cin; i += blockDim.x) sw[i] = w[i];
  for (int i = threadIdx.x; i < cout; i += blockDim.x) sw[kPwMaxCout * kPwMaxCin + i] = bias ? bias[i] : 0.f;
  __syncthreads();
  const int n = blockIdx.y;
  const __nv_bfloat16* xs = x + (long long)n * V * ld;
  float* ys = y + (long long)n * cout * V;
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < V; v += (long long)gridDim.x * blockDim.x) {
    float acc[kPwMaxCout];
#pragma unroll
    for (int o = 0; o < kPwMaxCout; ++o) acc[o] = sw[kPwMaxCout * kPwMaxCin + o];
    const __nv_bfloat16* xp = xs + v * ld;
    if constexpr (CIN > 0) {
      uint4 raw[CIN / 8];
#pragma unroll
      for (int c = 0; c < CIN / 8; ++c) raw[c] = __ldcs(reinterpret_cast<const uint4*>(xp) + c);
#pragma unroll
      for (int c = 0; c < CIN / 8; ++c) {
        float f[8];
        x16x8_to_float(raw[c], f, x_f16);
#pragma unroll
        for (int o = 0; o < kPwMaxCout; ++o)
          if (o < cout) {
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[o] = fmaf(f[i], sw[o * CIN + c * 8 + i], acc[o]);
          }
      }
    } else {
      for (int c0 = 0; c0 < cin; c0 += 8) {
        float f[8];
        x16x8_to_float(*reinterpret_cast<const uint4*>(xp + c0), f, x_f16);
#pragma unroll
        for (int o = 0; o < kPwMaxCout; ++o)
          if (o < cout) {
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[o] += f[i] * sw[o * cin + c0 + i];
          }
      }
    }
#pragma unroll
    for (int o = 0; o < kPwMaxCout; ++o)
      if (o < cout) __stcs(ys + (long long)o * V + v, acc[o]);
  }
}

// dx[v, ci] = sum_co dy[co, v] w[co][ci]; per-block partials of dw[co][ci] and dbias[co] into ws.
template <int kPwMaxCout>
__global__ void __launch_bounds__(256) pointwise_bwd_kernel(const __nv_bfloat16* x, long long ldx, const float* dy,
                                                            const float* w, __nv_bfloat16* dx, long long lddx, float* ws,
                                                            long long V, int cin, int cout, int x_f16) {
  __shared__ float sw[kPwMaxCout * kPwMaxCin];
  __shared__ float sacc[kPwMaxCout * (kPwMaxCin + 1)];
  for (int i = threadIdx.x; i < cout * cin; i += blockDim.x) sw[i] = w[i];
  for (int i = threadIdx.x; i < cout * (cin + 1); i += blockDim.x) sacc[i] = 0.f;
  __syncthreads();
  const int groups = cin / 8;
  const int n = blockIdx.y;  // sample: no 64-bit division in the voxel loop
  x += (long long)n * V * ldx;
  dy += (long long)n * cout * V;
  if (dx) dx += (long long)n * V * lddx;
  // thread = (voxel, channel group): keeps dw partials for its 8 channels x cout in registers
  float pw[kPwMaxCout][8];
  float pb[kPwMaxCout];
#pragma unroll
  for (int o = 0; o < kPwMaxCout; ++o) {
    pb[o] = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) pw[o][i] = 0.f;
  }
  // thread = (voxel lane, channel group): a thread always sees the same channel group
  const long long nthreads = (long long)gridDim.x * blockDim.x;
  const long long vlanes = nthreads / groups;
  const long long gtid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const int g = (int)(gtid % groups);
  const long long vlane = gtid / groups;
  // U voxels per iteration: all x loads and dy rows are issued before the arithmetic (the pass is bound by memory latency: 50 % of
  // the HBM peak with two voxels in flight per thread)
  constexpr int U = 4;
  for (long long vox = vlane; vlane < vlanes && vox < V; vox += U * vlanes) {
    uint4 r[U];
    float gy[U][kPwMaxCout];
    bool has[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long v = vox + u * vlanes;
      has[u] = v < V;
      r[u] = has[u] ? __ldcs(reinterpret_cast<const uint4*>(x + v * ldx + g * 8)) : make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int o = 0; o < kPwMaxCout; ++o) gy[u][o] = (o < cout && has[u]) ? dy[(long long)o * V + v] : 0.f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (!has[u]) break;
      const long long v = vox + u * vlanes;
      float f[8], d[8];
      x16x8_to_float(r[u], f, x_f16);
#pragma unroll
      for (int i = 0; i < 8; ++i) d[i] = 0.f;
#pragma unroll
      for (int o = 0; o < kPwMaxCout; ++o)
        if (o < cout) {
          if (g == 0) pb[o] += gy[u][o];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float wv = sw[o * cin + g * 8 + i];
            d[i] = fmaf(gy[u][o], wv, d[i]);
            pw[o][i] = fmaf(gy[u][o], f[i], pw[o][i]);
          }
        }
      if (dx) __stcs(reinterpret_cast<uint4*>(dx + v * lddx + g * 8), float_to_bf16x8(d));
    }
  }
  if (vlane < vlanes)
#pragma unroll
  for (int o = 0; o < kPwMaxCout; ++o)
    if (o < cout) {
#pragma unroll
      for (int i = 0; i < 8; ++i) atomicAdd(&sacc[o * (cin + 1) + g * 8 + i], pw[o][i]);
      if (g == 0) atomicAdd(&sacc[o * (cin + 1) + cin], pb[o]);
    }
  __syncthreads();
  const long long blk = (long long)blockIdx.y * gridDim.x + blockIdx.x;
  for (int i = threadIdx.x; i < cout * (cin + 1); i += blockDim.x) ws[blk * cout * (cin + 1) + i] = sacc[i];
}

// one block per output element: 256 threads stride through the per-block partials, shared-memory tree (double)
__global__ void __launch_bounds__(256) pointwise_bwd_reduce_kernel(const float* ws, int blocks, int cin, int cout, float* dw,
                                                                    float* dbias, int accumulate) {
  __shared__ double red[256];
  const int i = blockIdx.x;
  double s = 0.0;
  for (int b = threadIdx.x; b < blocks; b += 256) s += (double)ws[(long long)b * cout * (cin + 1) + i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int k = 128; k > 0; k >>= 1) {
    if (threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const float t = (float)red[0];
    const int o = i / (cin + 1), c = i % (cin + 1);
    if (c < cin) {
      if (dw) dw[o * cin + c] = accumulate ? dw[o * cin + c] + t : t;
    } else {
      if (dbias) dbias[o] = accumulate ? dbias[o] + t : t;
    }
  }
}

static int pointwise_bwd_blocks(const rehr_tensor* x) {  // per sample (grid.x); the launch uses grid.y = N
  const long long items = voxels_per_sample(x) * (x->c / 8);
  return std::max(1, grid_for(items, 256, 8) / std::max(1, x->n));
}

// per-channel sum over all voxels (bias gradient): per-block partials + reduce
__global__ void __launch_bounds__(256) channel_sum_kernel(const __nv_bfloat16* x, long long ld, long long total_vox, int C,
                                                          float* ws) {
  extern __shared__ float sh[];
  for (int i = threadIdx.x; i < C; i += blockDim.x) sh[i] = 0.f;
  __syncthreads();
  const int groups = C / 8;
  const long long items = total_vox * groups;
  const long long nthreads = (long long)gridDim.x * blockDim.x;
  const long long vlanes = nthreads / groups;
  const long long gtid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const int g = (int)(gtid % groups);
  const long long vlane = gtid / groups;
  (void)items;
  float s[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = 0.f;
  for (long long vox = vlane; vlane < vlanes && vox < total_vox; vox += vlanes) {
    float f[8];
    bf16x8_to_float(*reinterpret_cast<const uint4*>(x + vox * ld + g * 8), f);
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] += f[i];
  }
  if (vlane < vlanes) {
#pragma unroll
    for (int i = 0; i < 8; ++i) atomicAdd(&sh[g * 8 + i], s[i]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) ws[(long long)blockIdx.x * C + i] = sh[i];
}
// block = 32 channels x 8 slices of the partial list (fixed summation order -> deterministic)
__global__ void __launch_bounds__(256) channel_sum_reduce_kernel(const float* ws, int blocks, int C, float* out, int accumulate) {
  __shared__ double red[8][33];
  const int cl = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  double s = 0.0;
  if (c < C)
    for (int b = slice; b < blocks; b += 8) s += (double)ws[(long long)b * C + c];
  red[slice][cl] = s;
  __syncthreads();
  if (slice == 0 && c < C) {
    double t = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][cl];
    out[c] = accumulate ? out[c] + (float)t : (float)t;
  }
}
static int channel_sum_blocks(const rehr_tensor* x) {
  const long long items = (long long)x->n * voxels_per_sample(x) * (x->c / 8);
  return grid_for(items, 256, 4);
}

// =================================================================================================
// Depth-only linear upsampling, align_corners=True (ATen area_pixel_compute_source_index semantics)
// =================================================================================================
__global__ void __launch_bounds__(256) upsample_d_kernel(const __nv_bfloat16* x, long long ldx, __nv_bfloat16* y,
                                                         long long ldy, int N, int D, int OD, long long HW, int C, int x_f16,
                                                         int y_f16, RangeSlot* range) {
  const int groups = C / 8;
  const long long items = (long long)N * OD * HW * groups;
  const float scale = OD > 1 ? (float)(D - 1) / (float)(OD - 1) : 0.f;
  for (long long it = blockIdx.x * (long long)blockDim.x + threadIdx.x; it < items; it += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(it % groups);
    long long r = it / groups;
    const long long hw = r % HW;
    r /= HW;
    const int od = (int)(r % OD);
    const long long n = r / OD;
    const float src = scale * (float)od;
    const int i0 = (int)src;
    const int i1 = i0 + (i0 < D - 1 ? 1 : 0);
    const float l1 = src - (float)i0, l0 = 1.f - l1;
    float a[8], b[8], o[8];
    x16x8_to_float(*reinterpret_cast<const uint4*>(x + ((n * D + i0) * HW + hw) * ldx + g * 8), a, x_f16);
    x16x8_to_float(*reinterpret_cast<const uint4*>(x + ((n * D + i1) * HW + hw) * ldx + g * 8), b, x_f16);
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = l0 * a[i] + l1 * b[i];
    if (range != nullptr) range_check<8>(range, o);
    *reinterpret_cast<uint4*>(y + ((n * OD + od) * HW + hw) * ldy + g * 8) = float_to_x16x8(o, y_f16);
  }
}
// Source-centric variant: one thread per (n, source plane d, voxel, 8-channel group) loads planes d and d + 1 ONCE and writes every
// output plane whose lower source index is d (OD / D of them on average).  The output-centric kernel above re-read every source plane
// from DRAM ~3.4 times at the C4 shape (profiles/r02_ncu_families_raw.txt: 450 MB read for a 134 MB input).  Indices and weights come
// from the same float expressions, evaluated per output plane, so the results are bit-identical.
__global__ void __launch_bounds__(256) upsample_d_src_kernel(const __nv_bfloat16* x, long long ldx, __nv_bfloat16* y, long long ldy,
                                                             int N, int D, int OD, long long HW, int C, int x_f16, int y_f16,
                                                             RangeSlot* range) {
  const int groups = C / 8;
  const long long items = (long long)N * D * HW * groups;
  const float scale = OD > 1 ? (float)(D - 1) / (float)(OD - 1) : 0.f;
  for (long long it = blockIdx.x * (long long)blockDim.x + threadIdx.x; it < items; it += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(it % groups);
    long long r = it / groups;
    const long long hw = r % HW;
    r /= HW;
    const int d = (int)(r % D);
    const long long n = r / D;
    // first output plane with (int)(scale * od) >= d
    int od = 0;
    if (scale > 0.f) {
      od = max(0, min(OD - 1, (int)((float)d / scale) - 1));
      while (od > 0 && (int)(scale * (float)(od - 1)) >= d) --od;
      while (od < OD && (int)(scale * (float)od) < d) ++od;
    } else if (d > 0) {
      od = OD;  // every output plane reads source plane 0
    }
    if (od >= OD || (int)(scale * (float)od) != d) continue;
    float a[8], b[8], o[8];
    const int d1 = d + (d < D - 1 ? 1 : 0);
    x16x8_to_float(*reinterpret_cast<const uint4*>(x + ((n * D + d) * HW + hw) * ldx + g * 8), a, x_f16);
    x16x8_to_float(*reinterpret_cast<const uint4*>(x + ((n * D + d1) * HW + hw) * ldx + g * 8), b, x_f16);
    for (; od < OD; ++od) {
      const float src = scale * (float)od;
      const int i0 = (int)src;
      if (i0 != d) break;
      const float l1 = src - (float)i0, l0 = 1.f - l1;
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = l0 * a[i] + l1 * b[i];
      if (range != nullptr) range_check<8>(range, o);
      *reinterpret_cast<uint4*>(y + ((n * OD + od) * HW + hw) * ldy + g * 8) = float_to_x16x8(o, y_f16);
    }
  }
}
__global__ void __launch_bounds__(256) upsample_d_bwd_kernel(const __nv_bfloat16* dy, long long lddy, __nv_bfloat16* dx,
                                                             long long lddx, int N, int D, int OD, long long HW, int C) {
  const int groups = C / 8;
  const long long items = (long long)N * D * HW * groups;
  const float scale = OD > 1 ? (float)(D - 1) / (float)(OD - 1) : 0.f;
  for (long long it = blockIdx.x * (long long)blockDim.x + threadIdx.x; it < items; it += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(it % groups);
    long long r = it / groups;
    const long long hw = r % HW;
    r /= HW;
    const int d = (int)(r % D);
    const long long n = r / D;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    // output planes whose i0 or i1 equals d
    int j_lo = 0, j_hi = OD - 1;
    if (scale > 0.f) {
      j_lo = max(0, (int)floorf((float)(d - 1) / scale) - 1);
      j_hi = min(OD - 1, (int)ceilf((float)(d + 1) / scale) + 1);
    }
    for (int j = j_lo; j <= j_hi; ++j) {
      const float src = scale * (float)j;
      const int i0 = (int)src;
      const int i1 = i0 + (i0 < D - 1 ? 1 : 0);
      const float l1 = src - (float)i0, l0 = 1.f - l1;
      float wgt = 0.f;
      if (i0 == d) wgt += l0;
      if (i1 == d) wgt += l1;
      if (wgt != 0.f) {
        float f[8];
        bf16x8_to_float(*reinterpret_cast<const uint4*>(dy + ((n * OD + j) * HW + hw) * lddy + g * 8), f);
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] += wgt * f[i];
      }
    }
    *reinterpret_cast<uint4*>(dx + ((n * D + d) * HW + hw) * lddx + g * 8) = float_to_bf16x8(acc);
  }
}

// =================================================================================================
// Layout adapters: NCDHW f32 <-> NDHWC bf16 (32x32 shared-memory transpose per sample)
// =================================================================================================
__global__ void __launch_bounds__(256) ncdhw_to_ndhwc_kernel(const float* src, __nv_bfloat16* dst, long long ld, long long V,
                                                             int C) {
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const long long v0 = (long long)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int k = ty; k < 32; k += 8) {
    const int c = c0 + k;
    const long long v = v0 + tx;
    tile[k][tx] = (c < C && v < V) ? src[((long long)n * C + c) * V + v] : 0.f;
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const long long v = v0 + k;
    const int c = c0 + tx;
    if (c < C && v < V) dst[((long long)n * V + v) * ld + c] = __float2bfloat16(tile[tx][k]);
  }
}
__global__ void __launch_bounds__(256) ndhwc_to_ncdhw_kernel(const unsigned short* src, long long ld, float* dst, long long V,
                                                             int C, int src_f16) {
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const long long v0 = (long long)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int k = ty; k < 32; k += 8) {
    const long long v = v0 + k;
    const int c = c0 + tx;
    tile[k][tx] = (c < C && v < V) ? unpack16(src[((long long)n * V + v) * ld + c], src_f16) : 0.f;
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int c = c0 + k;
    const long long v = v0 + tx;
    if (c < C && v < V) dst[((long long)n * C + c) * V + v] = tile[tx][k];
  }
}

// 16-bit -> 16-bit format conversion of a (pitched) channels-last tensor: the bf16 twin of an fp16 forward activation that a
// weight-gradient GEMM needs as its operand (its other operand, the gradient, is bf16 and one MMA takes one format)
__global__ void __launch_bounds__(256) convert16_kernel(const __nv_bfloat16* x, long long ldx, int x_f16, __nv_bfloat16* y,
                                                        long long ldy, int y_f16, long long vox_total, int C, RangeSlot* range) {
  const int groups = C / 8;
  const long long items = vox_total * groups;
  for (long long it = blockIdx.x * (long long)blockDim.x + threadIdx.x; it < items; it += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(it % groups);
    const long long vox = it / groups;
    float f[8];
    x16x8_to_float(__ldcs(reinterpret_cast<const uint4*>(x + vox * ldx + g * 8)), f, x_f16);
    if (range != nullptr) range_check<8>(range, f);
    *reinterpret_cast<uint4*>(y + vox * ldy + g * 8) = float_to_x16x8(f, y_f16);
  }
}

// =================================================================================================
// SE-gate tail: y = act(x * gate[n,c] (+ residual))
// =================================================================================================
__global__ void __launch_bounds__(256) segate_kernel(const __nv_bfloat16* x, long long ldx, const float* gate,
                                                     const __nv_bfloat16* res, long long ldr, __nv_bfloat16* y,
                                                     long long ldy, int N, long long V, int C, int act, float slope) {
  const int groups = C / 8;
  const long long items = (long long)N * V * groups;
  for (long long it = blockIdx.x * (long long)blockDim.x + threadIdx.x; it < items; it += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(it % groups);
    const long long vox = it / groups;
    const long long n = vox / V;
    float f[8], o[8];
    bf16x8_to_float(*reinterpret_cast<const uint4*>(x + vox * ldx + g * 8), f);
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = f[i] * (gate ? gate[n * C + g * 8 + i] : 1.f);
    if (res) {
      float r[8];
      bf16x8_to_float(*reinterpret_cast<const uint4*>(res + vox * ldr + g * 8), r);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] += r[i];
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (act == REHR_ACT_RELU) o[i] = o[i] > 0.f ? o[i] : 0.f;
      if (act == REHR_ACT_LRELU) o[i] = o[i] > 0.f ? o[i] : o[i] * slope;
    }
    *reinterpret_cast<uint4*>(y + vox * ldy + g * 8) = float_to_bf16x8(o);
  }
}

// SE-gate tail backward.  With m = act'(y) evaluated from the OUTPUT y (ReLU / LeakyReLU slope > 0 / none) and g = dy * m:
//   reduce:  partial[n][tile][c] = (sum_v g * x, 0)                      -> d(gate)[n,c]
//   apply :  dx = g * gate[n,c] + shift[n,c]   (shift = d(pool)/V, the gradient through the global average pool)
//            dres = g (optional)
template <int MODE>  // 0 reduce, 1 apply
__global__ void __launch_bounds__(kStatThreads) segate_bwd_kernel(const __nv_bfloat16* x, long long ldx, const __nv_bfloat16* y,
                                                                  long long ldy, const __nv_bfloat16* dy, long long lddy,
                                                                  const float* gate, const float* shift, __nv_bfloat16* dx,
                                                                  long long lddx, __nv_bfloat16* dres, long long lddr,
                                                                  float* partial, long long V, int C, int tiles, int vpb, int act,
                                                                  float slope) {
  extern __shared__ float sh[];
  const int n = blockIdx.y, tile = blockIdx.x;
  const int groups = C / 8;
  const int lanes = kStatThreads / groups;
  const int g = threadIdx.x % groups, vl = threadIdx.x / groups;
  const long long v0 = (long long)tile * vpb, v1 = min(V, v0 + vpb);
  float acc[8], ga[8], sf[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    acc[i] = 0.f;
    ga[i] = (MODE == 1 && gate) ? gate[n * C + g * 8 + i] : 1.f;
    sf[i] = (MODE == 1 && shift) ? shift[n * C + g * 8 + i] : 0.f;
  }
  if (vl < lanes) {
    for (long long v = v0 + vl; v < v1; v += lanes) {
      const long long vox = (long long)n * V + v;
      float d[8];
      bf16x8_to_float(*reinterpret_cast<const uint4*>(dy + vox * lddy + g * 8), d);
      if (act != REHR_ACT_NONE) {
        float yy[8];
        bf16x8_to_float(*reinterpret_cast<const uint4*>(y + vox * ldy + g * 8), yy);
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (!(yy[i] > 0.f)) d[i] *= (act == REHR_ACT_LRELU ? slope : 0.f);
      }
      if (MODE == 0) {
        float xx[8];
        bf16x8_to_float(*reinterpret_cast<const uint4*>(x + vox * ldx + g * 8), xx);
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = fmaf(d[i], xx[i], acc[i]);
      } else {
        float o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = fmaf(d[i], ga[i], sf[i]);
        *reinterpret_cast<uint4*>(dx + vox * lddx + g * 8) = float_to_bf16x8(o);
        if (dres) *reinterpret_cast<uint4*>(dres + vox * lddr + g * 8) = float_to_bf16x8(d);
      }
    }
  }
  if (MODE == 0) {
    if (vl < lanes) {
#pragma unroll
      for (int i = 0; i < 8; ++i) sh[vl * C + g * 8 + i] = acc[i];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += kStatThreads) {
      float t = 0.f;
      for (int l = 0; l < lanes; ++l) t += sh[l * C + c];
      float* dst = partial + (((long long)n * tiles + tile) * C + c) * 2;
      dst[0] = t;
      dst[1] = 0.f;
    }
  }
}

// =================================================================================================
// Sliding-window Gaussian blend with fp16 accumulators (bit-faithful to ATen half arithmetic:
// every half op computes in float and rounds once).
// =================================================================================================
__global__ void __launch_bounds__(256) sw_accumulate_kernel(__half* logits, __half* npred, const void* pred, int pred_f32,
                                                            const __half* gauss, int C, int VD, int VH, int VW, int TD,
                                                            int TH, int TW, int od, int oh, int ow) {
  const long long tv = (long long)TD * TH * TW;
  const long long vv = (long long)VD * VH * VW;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < tv; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % TW);
    const int y = (int)((i / TW) % TH);
    const int z = (int)(i / ((long long)TW * TH));
    const long long vi = ((long long)(od + z) * VH + (oh + y)) * VW + (ow + x);
    const float g = gauss ? __half2float(gauss[i]) : 1.f;
    for (int c = 0; c < C; ++c) {
      // ATen semantics of `logits[sl] += pred * gauss` (utils/seg_utils.py:275): a half x half product is rounded to half
      // before the add; a float prediction promotes the product and the add to float, rounding once at the store.
      float prod;
      if (pred_f32)
        prod = __fmul_rn(reinterpret_cast<const float*>(pred)[c * tv + i], g);  // rounded product, never contracted into an FMA
      else
        prod = __half2float(__float2half(__half2float(reinterpret_cast<const __half*>(pred)[c * tv + i]) * g));
      logits[c * vv + vi] = __float2half(__half2float(logits[c * vv + vi]) + prod);
    }
    if (npred) npred[vi] = __float2half(__half2float(npred[vi]) + g);
  }
}
__global__ void __launch_bounds__(256) sw_finalize_kernel(__half* logits, const __half* npred, int C, long long vv,
                                                          int* inf_flag) {
  int bad = 0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < vv; i += (long long)gridDim.x * blockDim.x) {
    const float n = __half2float(npred[i]);
    for (int c = 0; c < C; ++c) {
      const __half q = __float2half(__half2float(logits[c * vv + i]) / n);
      logits[c * vv + i] = q;
      if (__hisinf(q)) bad = 1;
    }
  }
  if (bad && inf_flag) atomicOr(inf_flag, 1);
}

// 16-byte variants (tile width, x offset and volume width multiples of 8, 16-byte aligned bases): eight voxels of a row per thread,
// the per-element arithmetic (and therefore every rounding) exactly as in the scalar kernels above.
__device__ __forceinline__ void half8_unpack(const uint4& u, float (&f)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = __half22float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 half8_pack(const __half (&h)[8]) {
  uint4 u;
  __half2* o = reinterpret_cast<__half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) o[i] = __halves2half2(h[2 * i], h[2 * i + 1]);
  return u;
}
__global__ void __launch_bounds__(256) sw_accumulate_vec8_kernel(__half* logits, __half* npred, const void* pred, int pred_f32,
                                                                 const __half* gauss, int C, int VD, int VH, int VW, int TD,
                                                                 int TH, int TW, int od, int oh, int ow) {
  const int TW8 = TW / 8;
  const long long groups = (long long)TD * TH * TW8;
  const long long tv = (long long)TD * TH * TW;
  const long long vv = (long long)VD * VH * VW;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < groups; q += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(q % TW8) * 8;
    const int y = (int)((q / TW8) % TH);
    const int z = (int)(q / ((long long)TW8 * TH));
    const long long i = ((long long)z * TH + y) * TW + x;
    const long long vi = ((long long)(od + z) * VH + (oh + y)) * VW + (ow + x);
    float g[8];
    if (gauss) {
      half8_unpack(*reinterpret_cast<const uint4*>(gauss + i), g);
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) g[e] = 1.f;
    }
    for (int c = 0; c < C; ++c) {
      float prod[8], acc[8];
      if (pred_f32) {
        const float4* pp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(pred) + c * tv + i);
        const float4 a = pp[0], b = pp[1];
        prod[0] = __fmul_rn(a.x, g[0]); prod[1] = __fmul_rn(a.y, g[1]); prod[2] = __fmul_rn(a.z, g[2]); prod[3] = __fmul_rn(a.w, g[3]);
        prod[4] = __fmul_rn(b.x, g[4]); prod[5] = __fmul_rn(b.y, g[5]); prod[6] = __fmul_rn(b.z, g[6]); prod[7] = __fmul_rn(b.w, g[7]);
      } else {
        float pv[8];
        half8_unpack(*reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(pred) + c * tv + i), pv);
#pragma unroll
        for (int e = 0; e < 8; ++e) prod[e] = __half2float(__float2half(pv[e] * g[e]));
      }
      uint4* lp = reinterpret_cast<uint4*>(logits + c * vv + vi);
      half8_unpack(*lp, acc);
      __half r[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) r[e] = __float2half(acc[e] + prod[e]);
      *lp = half8_pack(r);
    }
    if (npred) {
      uint4* np = reinterpret_cast<uint4*>(npred + vi);
      float a[8];
      half8_unpack(*np, a);
      __half r[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) r[e] = __float2half(a[e] + g[e]);
      *np = half8_pack(r);
    }
  }
}
__global__ void __launch_bounds__(256) sw_finalize_vec8_kernel(__half* logits, const __half* npred, int C, long long vv,
                                                               int* inf_flag) {
  int bad = 0;
  const long long groups = vv / 8;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < groups; q += (long long)gridDim.x * blockDim.x) {
    float n[8];
    half8_unpack(*reinterpret_cast<const uint4*>(npred + q * 8), n);
    for (int c = 0; c < C; ++c) {
      uint4* lp = reinterpret_cast<uint4*>(logits + c * vv + q * 8);
      float a[8];
      half8_unpack(*lp, a);
      __half r[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        r[e] = __float2half(a[e] / n[e]);
        if (__hisinf(r[e])) bad = 1;
      }
      *lp = half8_pack(r);
    }
  }
  if (bad && inf_flag) atomicOr(inf_flag, 1);
}

// =================================================================================================
// Blur degradation: L-tap cross-correlation along X of x[Z][X][Y] (F.conv2d padding="same")
// =================================================================================================
static constexpr int kBlurMaxTaps = 65;
struct BlurTaps {
  float t[kBlurMaxTaps];
};
// Tile = kBlurRows output rows (along X) x 128 columns (along Y, the contiguous axis): the kBlurRows + L - 1 input rows are
// staged once in shared memory with coalesced 512 B row reads, every thread then slides down its column (bank-conflict free),
// so each input element is read from HBM ~(1 + (L-1)/kBlurRows) times instead of L times through L2.
static constexpr int kBlurRows = 64;
__global__ void __launch_bounds__(128) blur1d_kernel(const float* x, float* y, const float* taps, int L, long long Z, int X,
                                                     int Y) {
  extern __shared__ float tile[];  // [kBlurRows + L - 1][128]
  __shared__ float st[kBlurMaxTaps];
  for (int i = threadIdx.x; i < L; i += blockDim.x) st[i] = taps[i];
  const int left = (L - 1) / 2;
  const int ytiles = (Y + 127) / 128, xtiles = (X + kBlurRows - 1) / kBlurRows;
  const long long total = Z * (long long)xtiles * ytiles;
  const int rows_in = kBlurRows + L - 1;
  for (long long t = blockIdx.x; t < total; t += gridDim.x) {
    const int yt = (int)(t % ytiles);
    const int xt = (int)((t / ytiles) % xtiles);
    const long long z = t / ((long long)ytiles * xtiles);
    const int yy = yt * 128 + threadIdx.x;
    const int x0 = xt * kBlurRows;
    const float* base = x + z * (long long)X * Y;
    __syncthreads();
    for (int r = 0; r < rows_in; ++r) {
      const int xs = x0 + r - left;
      tile[r * 128 + threadIdx.x] = (xs >= 0 && xs < X && yy < Y) ? base[(long long)xs * Y + yy] : 0.f;
    }
    __syncthreads();
    if (yy < Y) {
      float* out = y + z * (long long)X * Y;
      const int nrows = min(kBlurRows, X - x0);
      for (int r = 0; r < nrows; ++r) {
        float acc = 0.f;
        for (int l = 0; l < L; ++l) acc += st[l] * tile[(r + l) * 128 + threadIdx.x];
        out[(long long)(x0 + r) * Y + yy] = acc;
      }
    }
  }
}

// Same tile, 16-byte accesses (Y % 4 == 0, 16-byte aligned bases): a warp stages one 512 B row per load instruction with several rows
// in flight, then every thread owns a 4-column strip of kBlurRows / 4 output rows and computes them four at a time -- each staged
// float4 feeds the (up to) four outputs it belongs to, taps applied in ascending order exactly like the scalar kernel (bit-identical
// results), one LDS.128 per staged row instead of one per tap.
__global__ void __launch_bounds__(128) blur1d_vec4_kernel(const float* __restrict__ x, float* __restrict__ y, const float* __restrict__ taps,
                                                          int L, long long Z, int X, int Y) {
  extern __shared__ float tile[];  // [kBlurRows + L - 1][128]
  __shared__ float st[kBlurMaxTaps];
  for (int i = threadIdx.x; i < L; i += blockDim.x) st[i] = taps[i];
  const int left = (L - 1) / 2;
  const int ytiles = (Y + 127) / 128, xtiles = (X + kBlurRows - 1) / kBlurRows;
  const long long total = Z * (long long)xtiles * ytiles;
  const int rows_in = kBlurRows + L - 1;
  const int cq = threadIdx.x & 31, rr = threadIdx.x >> 5;  // column quad, row phase
  constexpr int kStrip = kBlurRows / 4;                    // output rows per thread
  float4* tile4 = reinterpret_cast<float4*>(tile);         // [rows_in][32]
  for (long long t = blockIdx.x; t < total; t += gridDim.x) {
    const int yt = (int)(t % ytiles);
    const int xt = (int)((t / ytiles) % xtiles);
    const long long z = t / ((long long)ytiles * xtiles);
    const int yy = yt * 128 + cq * 4;
    const int x0 = xt * kBlurRows;
    const float* base = x + z * (long long)X * Y;
    const bool col_ok = yy < Y;  // Y % 4 == 0: the quad is inside or outside as a whole
    __syncthreads();
#pragma unroll 6
    for (int r = rr; r < rows_in; r += 4) {
      const int xs = x0 + r - left;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (col_ok && xs >= 0 && xs < X) v = *reinterpret_cast<const float4*>(base + (long long)xs * Y + yy);
      tile4[r * 32 + cq] = v;
    }
    __syncthreads();
    if (col_ok) {
      float* out = y + z * (long long)X * Y;
      const int nrows = min(kBlurRows, X - x0);
      for (int r0 = rr * kStrip; r0 < min(nrows, (rr + 1) * kStrip); r0 += 4) {
        float4 acc[4];
#pragma unroll
        for (int o = 0; o < 4; ++o) acc[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        float w0 = 0.f, w1 = 0.f, w2 = 0.f, w3 = 0.f;  // taps j, j-1, j-2, j-3
        for (int j = 0; j < L + 3; ++j) {
          w3 = w2;
          w2 = w1;
          w1 = w0;
          w0 = j < L ? st[j] : 0.f;
          const float4 v = tile4[(r0 + j) * 32 + cq];  // r0 + j <= r0 + L + 2 <= kBlurRows + L - 2: inside the staged tile
          if (j < L) {
            acc[0].x += w0 * v.x; acc[0].y += w0 * v.y; acc[0].z += w0 * v.z; acc[0].w += w0 * v.w;
          }
          if (j >= 1 && j - 1 < L) {
            acc[1].x += w1 * v.x; acc[1].y += w1 * v.y; acc[1].z += w1 * v.z; acc[1].w += w1 * v.w;
          }
          if (j >= 2 && j - 2 < L) {
            acc[2].x += w2 * v.x; acc[2].y += w2 * v.y; acc[2].z += w2 * v.z; acc[2].w += w2 * v.w;
          }
          if (j >= 3) {
            acc[3].x += w3 * v.x; acc[3].y += w3 * v.y; acc[3].z += w3 * v.z; acc[3].w += w3 * v.w;
          }
        }
#pragma unroll
        for (int o = 0; o < 4; ++o)
          if (r0 + o < nrows) *reinterpret_cast<float4*>(out + (long long)(x0 + r0 + o) * Y + yy) = acc[o];
      }
    }
  }
}

// =================================================================================================
// rot90 over dims (0,1) of vol[X][Y][inner], torch.rot90 semantics
// =================================================================================================
// -------------------------------------------------------------------------------------------------
// Order-3 spline resampling of 2-D slices under an affine map: the stage-2 spatial augmentation (rotation / scaling of every slice of
// a patch, `augment_spatial` -> batchgenerators `interpolate_img` -> scipy.ndimage.map_coordinates, utils/seg_utils.py:378-458).
// scipy's order-3 interpolation = (1) cubic B-spline prefilter of the image along each axis (one causal + one anti-causal
// recursion with the pole z = sqrt(3) - 2 and MIRROR boundary initialisation, gain 6), (2) evaluation of the 4 x 4 B-spline taps
// around the sample position with mirrored tap indices; mode "constant": positions outside [0, n - 1] give cval.
// -------------------------------------------------------------------------------------------------
// in place along the middle axis of c[outer][n][inner]; one thread per line
__global__ void __launch_bounds__(128) bspline_prefilter_kernel(float* __restrict__ c, long long outer, int n, long long inner) {
  const long long line = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (line >= outer * inner || n < 2) return;
  bspline_prefilter_line(c + (line / inner) * (long long)n * inner + (line % inner), n, inner);
}

struct AffineSampleArgs {
  const float* src;     // [S][X][Y]: B-spline coefficients (order 3) or the image itself (order 1 / labels)
  float* dst;           // [S][PX][PY]
  const float* affine;  // [samples][6]: a00 a01 a10 a11 cx cy   (source position = A * (i - (PX-1)/2, j - (PY-1)/2) + c)
  int S, X, Y, PX, PY, per_sample;  // slices per sample (slice s uses affine[s / per_sample])
  int order;            // 3: cubic B-spline of coefficients; 1: per-label linear interpolation (is_seg)
  float cval;
  int n_labels;
  float labels[8];      // order 1: ascending label values; the result is the LAST label whose interpolated indicator is >= 0.5
};

__device__ __forceinline__ int mirror_idx(int i, int n) {
  if (n == 1) return 0;
  const int period = 2 * (n - 1);
  i = abs(i) % period;
  return i < n ? i : period - i;
}

__global__ void __launch_bounds__(256) affine_sample2d_kernel(const AffineSampleArgs a) {
  const long long total = (long long)a.S * a.PX * a.PY;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(e % a.PY);
    const long long t = e / a.PY;
    const int i = (int)(t % a.PX);
    const int s = (int)(t / a.PX);
    const float* A = a.affine + (long long)(s / a.per_sample) * 6;
    // double precision for the position (the reference computes it in fp64; an fp32 position moves a sample by up to 3e-5 pixels)
    const double mi = (double)i - 0.5 * (double)(a.PX - 1), mj = (double)j - 0.5 * (double)(a.PY - 1);
    const double x = (double)A[0] * mi + (double)A[1] * mj + (double)A[4];
    const double y = (double)A[2] * mi + (double)A[3] * mj + (double)A[5];
    const float* img = a.src + (long long)s * a.X * a.Y;
    float out;
    if (x < 0.0 || x > (double)(a.X - 1) || y < 0.0 || y > (double)(a.Y - 1)) {
      out = a.order == 3 ? a.cval : 0.f;        // labels: an all-cval (-1) sample never reaches 0.5 -> the zero initialisation stays
    } else if (a.order == 3) {
      const int fx = (int)floor(x), fy = (int)floor(y);
      const float tx = (float)(x - (double)fx), ty = (float)(y - (double)fy);
      float wx[4], wy[4];
      wx[0] = (1.f - tx) * (1.f - tx) * (1.f - tx) * (1.f / 6.f);
      wx[1] = (3.f * tx * tx * tx - 6.f * tx * tx + 4.f) * (1.f / 6.f);
      wx[2] = (-3.f * tx * tx * tx + 3.f * tx * tx + 3.f * tx + 1.f) * (1.f / 6.f);
      wx[3] = tx * tx * tx * (1.f / 6.f);
      wy[0] = (1.f - ty) * (1.f - ty) * (1.f - ty) * (1.f / 6.f);
      wy[1] = (3.f * ty * ty * ty - 6.f * ty * ty + 4.f) * (1.f / 6.f);
      wy[2] = (-3.f * ty * ty * ty + 3.f * ty * ty + 3.f * ty + 1.f) * (1.f / 6.f);
      wy[3] = ty * ty * ty * (1.f / 6.f);
      float v = 0.f;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const float* row = img + (long long)mirror_idx(fx - 1 + p, a.X) * a.Y;
        float r = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) r += wy[q] * row[mirror_idx(fy - 1 + q, a.Y)];
        v += wx[p] * r;
      }
      out = v;
    } else {
      const int fx = (int)floor(x), fy = (int)floor(y);
      const float tx = (float)(x - (double)fx), ty = (float)(y - (double)fy);
      const int x1 = mirror_idx(fx + 1, a.X), y1 = mirror_idx(fy + 1, a.Y);
      const float v00 = img[(long long)fx * a.Y + fy], v01 = img[(long long)fx * a.Y + y1];
      const float v10 = img[(long long)x1 * a.Y + fy], v11 = img[(long long)x1 * a.Y + y1];
      out = 0.f;
      for (int l = 0; l < a.n_labels; ++l) {
        const float c = a.labels[l];
        const float ind = (1.f - tx) * ((1.f - ty) * (v00 == c ? 1.f : 0.f) + ty * (v01 == c ? 1.f : 0.f)) +
                          tx * ((1.f - ty) * (v10 == c ? 1.f : 0.f) + ty * (v11 == c ? 1.f : 0.f));
        if (ind >= 0.5f) out = c;
      }
    }
    a.dst[e] = out;
  }
}

// -------------------------------------------------------------------------------------------------
// UASR head of the FLAVR network (models/FLAVR/FLAVR_arch.py:203-227,244-246): per pixel and output slice, a softmax over
// E = 16 experts mixes the experts' image / segmentation predictions and gives the uncertainty:
//   p = softmax(ue[0..E)),  img = sum_e p_e (tanh(o[2e]) + 1) / 2,  seg = sum_e p_e o[2e+1],  unc = sigmoid(sum_e p_e w_e + b).
// The reference spells this as ~10 PyTorch passes over [B, 32, n_out, H, W] fp32 tensors; here one pass reads the two conv outputs
// where they lie (channels-last fp32 [pixel][slice*2E + c] and [pixel][slice*E + e]) and writes NCDHW results.
// -------------------------------------------------------------------------------------------------
static constexpr int kUasrE = 16;

struct UasrArgs {
  const float* out;   // [pixels][n_out * 2E]
  const float* ue;    // [pixels][n_out * E]
  const float* w;     // [E]
  const float* b;     // [1]
  float* res;         // [B][2][n_out][HW]
  float* unc;         // [B][1][n_out][HW]
  const float* d_res; // backward
  const float* d_unc;
  float* d_out;       // [pixels][n_out * 2E]
  float* d_ue;        // [pixels][n_out * E]
  float* partial;     // [blocks][E + 1]: per-block sums of d_u * p_e and of d_u
  long long pixels, HW;
  int n_out;
};

__device__ __forceinline__ void uasr_load(const UasrArgs& a, long long px, int o, float (&x)[2 * kUasrE], float (&p)[kUasrE]) {
  const float4* po = reinterpret_cast<const float4*>(a.out + (px * a.n_out + o) * (2 * kUasrE));
  const float4* pu = reinterpret_cast<const float4*>(a.ue + (px * a.n_out + o) * kUasrE);
#pragma unroll
  for (int i = 0; i < 2 * kUasrE / 4; ++i) {
    const float4 v = __ldg(po + i);
    x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
  }
  float m = -3.4e38f;
#pragma unroll
  for (int i = 0; i < kUasrE / 4; ++i) {
    const float4 v = __ldg(pu + i);
    p[4 * i] = v.x; p[4 * i + 1] = v.y; p[4 * i + 2] = v.z; p[4 * i + 3] = v.w;
  }
#pragma unroll
  for (int e = 0; e < kUasrE; ++e) m = fmaxf(m, p[e]);
  float sum = 0.f;
#pragma unroll
  for (int e = 0; e < kUasrE; ++e) {
    p[e] = expf(p[e] - m);
    sum += p[e];
  }
  const float inv = 1.f / sum;
#pragma unroll
  for (int e = 0; e < kUasrE; ++e) p[e] *= inv;
}

__global__ void __launch_bounds__(128) uasr_mixture_fwd_kernel(const UasrArgs a) {
  __shared__ float sw[kUasrE + 1];
  if (threadIdx.x <= kUasrE) sw[threadIdx.x] = threadIdx.x < kUasrE ? a.w[threadIdx.x] : a.b[0];
  __syncthreads();
  const long long total = a.pixels * a.n_out;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int o = (int)(t / a.pixels);          // slice-major: consecutive threads = consecutive pixels (coalesced NCDHW stores)
    const long long px = t - (long long)o * a.pixels;
    float x[2 * kUasrE], p[kUasrE];
    uasr_load(a, px, o, x, p);
    float img = 0.f, seg = 0.f, u = sw[kUasrE];
#pragma unroll
    for (int e = 0; e < kUasrE; ++e) {
      img = fmaf(p[e], 0.5f * (tanhf(x[2 * e]) + 1.f), img);
      seg = fmaf(p[e], x[2 * e + 1], seg);
      u = fmaf(p[e], sw[e], u);
    }
    const long long bidx = px / a.HW, hw = px - bidx * a.HW;
    a.res[((bidx * 2 + 0) * a.n_out + o) * a.HW + hw] = img;
    a.res[((bidx * 2 + 1) * a.n_out + o) * a.HW + hw] = seg;
    a.unc[(bidx * a.n_out + o) * a.HW + hw] = 1.f / (1.f + expf(-u));
  }
}

__global__ void __launch_bounds__(128) uasr_mixture_bwd_kernel(const UasrArgs a) {
  __shared__ float sw[kUasrE + 1];
  __shared__ float sred[4][kUasrE + 1];
  if (threadIdx.x <= kUasrE) sw[threadIdx.x] = threadIdx.x < kUasrE ? a.w[threadIdx.x] : a.b[0];
  __syncthreads();
  float aw[kUasrE + 1];
#pragma unroll
  for (int e = 0; e <= kUasrE; ++e) aw[e] = 0.f;
  const long long total = a.pixels * a.n_out;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int o = (int)(t / a.pixels);
    const long long px = t - (long long)o * a.pixels;
    float x[2 * kUasrE], p[kUasrE];
    uasr_load(a, px, o, x, p);
    const long long bidx = px / a.HW, hw = px - bidx * a.HW;
    const float d_img = a.d_res ? a.d_res[((bidx * 2 + 0) * a.n_out + o) * a.HW + hw] : 0.f;
    const float d_seg = a.d_res ? a.d_res[((bidx * 2 + 1) * a.n_out + o) * a.HW + hw] : 0.f;
    float u = sw[kUasrE];
#pragma unroll
    for (int e = 0; e < kUasrE; ++e) u = fmaf(p[e], sw[e], u);
    const float s = 1.f / (1.f + expf(-u));
    const float d_u = a.d_unc ? a.d_unc[(bidx * a.n_out + o) * a.HW + hw] * s * (1.f - s) : 0.f;
    float q[kUasrE], dx[2 * kUasrE];
    float pq = 0.f;
#pragma unroll
    for (int e = 0; e < kUasrE; ++e) {
      const float th = tanhf(x[2 * e]);
      q[e] = d_img * 0.5f * (th + 1.f) + d_seg * x[2 * e + 1] + d_u * sw[e];
      pq = fmaf(p[e], q[e], pq);
      dx[2 * e] = d_img * p[e] * 0.5f * (1.f - th * th);
      dx[2 * e + 1] = d_seg * p[e];
      aw[e] = fmaf(d_u, p[e], aw[e]);
    }
    aw[kUasrE] += d_u;
    float4* po = reinterpret_cast<float4*>(a.d_out + (px * a.n_out + o) * (2 * kUasrE));
#pragma unroll
    for (int i = 0; i < 2 * kUasrE / 4; ++i) po[i] = make_float4(dx[4 * i], dx[4 * i + 1], dx[4 * i + 2], dx[4 * i + 3]);
    float4* pu = reinterpret_cast<float4*>(a.d_ue + (px * a.n_out + o) * kUasrE);
#pragma unroll
    for (int i = 0; i < kUasrE / 4; ++i)
      pu[i] = make_float4(p[4 * i] * (q[4 * i] - pq), p[4 * i + 1] * (q[4 * i + 1] - pq), p[4 * i + 2] * (q[4 * i + 2] - pq),
                          p[4 * i + 3] * (q[4 * i + 3] - pq));
  }
  // per-block sums of the uncertainty layer's gradients (fixed order: warp shuffle, then the 4 warps)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int e = 0; e <= kUasrE; ++e) {
    float v = aw[e];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if (lane == 0) sred[warp][e] = v;
  }
  __syncthreads();
  if (threadIdx.x <= kUasrE)
    a.partial[(long long)blockIdx.x * (kUasrE + 1) + threadIdx.x] = sred[0][threadIdx.x] + sred[1][threadIdx.x] + sred[2][threadIdx.x] + sred[3][threadIdx.x];
}

// Resampling along ONE axis of x[outer][n_in][inner] -> y[outer][n_out][inner] with step `d` and the same field of view: output
// sample i sits at p = (i + 0.5) * d - 0.5 input samples.  order 3: cubic convolution (A = -0.75, the kernel of torch's bicubic
// grid_sample) over the 4 neighbours floor(p) - 1 .. floor(p) + 2 with indices clamped to the volume; order 0: nearest
// (floor(p + 0.5), clamped).  The low-resolution simulation of the SR stage, `resize(img, (slice_separation, 1), order)` at
// utils/train_set.py:395-396 -- the third-party `resize` package is not available, this is the stand-in oracle/degrade.py defines.
__global__ void __launch_bounds__(256) resample_axis_kernel(const float* __restrict__ x, float* __restrict__ y, long long outer, int n_in,
                                                            int n_out, long long inner, float d, int order) {
  const long long total = outer * n_out * inner;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e % inner;
    const long long t = e / inner;
    const int i = (int)(t % n_out);
    const long long o = t / n_out;
    const float p = ((float)i + 0.5f) * d - 0.5f;
    const float* src = x + o * n_in * inner + r;
    float v;
    if (order == 0) {
      int j = (int)floorf(p + 0.5f);
      j = min(max(j, 0), n_in - 1);
      v = src[(long long)j * inner];
    } else {
      const float fl = floorf(p);
      const float f = p - fl;
      const int j0 = (int)fl;
      const float A = -0.75f;
      const float w0 = ((A * (f + 1.f) - 5.f * A) * (f + 1.f) + 8.f * A) * (f + 1.f) - 4.f * A;
      const float w1 = ((A + 2.f) * f - (A + 3.f)) * f * f + 1.f;
      const float g = 1.f - f;
      const float w2 = ((A + 2.f) * g - (A + 3.f)) * g * g + 1.f;
      const float w3 = ((A * (g + 1.f) - 5.f * A) * (g + 1.f) + 8.f * A) * (g + 1.f) - 4.f * A;
      const int a0 = min(max(j0 - 1, 0), n_in - 1), a1 = min(max(j0, 0), n_in - 1);
      const int a2 = min(max(j0 + 1, 0), n_in - 1), a3 = min(max(j0 + 2, 0), n_in - 1);
      v = w0 * src[(long long)a0 * inner] + w1 * src[(long long)a1 * inner] + w2 * src[(long long)a2 * inner] + w3 * src[(long long)a3 * inner];
    }
    y[e] = v;
  }
}

template <typename T>
__global__ void __launch_bounds__(256) rot90_kernel(const T* src, T* dst, int X, int Y, long long inner, int k) {
  const int OX = (k & 1) ? Y : X, OY = (k & 1) ? X : Y;
  const long long total = (long long)OX * OY * inner;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long e = i % inner;
    const long long ij = i / inner;
    const int j = (int)(ij % OY), ii = (int)(ij / OY);
    int sx, sy;
    if (k == 1) {
      sx = j;
      sy = Y - 1 - ii;
    } else if (k == 2) {
      sx = X - 1 - ii;
      sy = Y - 1 - j;
    } else {  // k == 3
      sx = X - 1 - j;
      sy = ii;
    }
    dst[i] = src[((long long)sx * Y + sy) * inner + e];
  }
}

// =================================================================================================
// FBA spectral combine and orientation mean
// =================================================================================================
static constexpr int kMaxFuse = 16;
struct PtrPack {
  const void* p[kMaxFuse];
};
// One spectral bin: the K values of that bin sit in registers (KMAX = 4 / 8 / 16, loops fully unrolled and predicated on k < K).
template <int KMAX>
__device__ __forceinline__ float2 fba_bin(const float2 (&v)[KMAX], int K, float p) {
  if (p < 0.f) {
    // numpy max on complex: lexicographic (real, then imag); NaN propagates like np.maximum
    float2 best = v[0];
#pragma unroll
    for (int k = 1; k < KMAX; ++k) {
      if (k < K) {
        const bool best_nan = (best.x != best.x) || (best.y != best.y);
        const bool v_nan = (v[k].x != v[k].x) || (v[k].y != v[k].y);
        if (!best_nan && (v_nan || v[k].x > best.x || (v[k].x == best.x && v[k].y > best.y))) best = v[k];
      }
    }
    return best;
  }
  float mag[KMAX];
  float den = 0.f;
#pragma unroll
  for (int k = 0; k < KMAX; ++k) {
    if (k < K) {
      mag[k] = powf(hypotf(v[k].x, v[k].y), p);
      den += mag[k];
    }
  }
  float2 acc = make_float2(0.f, 0.f);
#pragma unroll
  for (int k = 0; k < KMAX; ++k) {
    if (k < K) {
      const float w = mag[k] / den;
      acc.x += w * v[k].x;
      acc.y += w * v[k].y;
    }
  }
  return acc;
}
// V = bins per thread: 2 (one 16-byte access per spectrum; even bin count, 16-byte aligned bases) or 1.  All K loads of a thread are
// issued before the first use.
template <int KMAX, int V>
__global__ void __launch_bounds__(256) fba_combine_kernel(PtrPack sp, int K, float p, float2* out, long long n) {
  const long long items = n / V;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < items; i += (long long)gridDim.x * blockDim.x) {
    float2 a[KMAX], b[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
      if (k < K) {
        if (V == 2) {
          const float4 t = reinterpret_cast<const float4*>(sp.p[k])[i];
          a[k] = make_float2(t.x, t.y);
          b[k] = make_float2(t.z, t.w);
        } else {
          a[k] = reinterpret_cast<const float2*>(sp.p[k])[i];
        }
      }
    }
    if (V == 2) {
      const float2 r0 = fba_bin<KMAX>(a, K, p), r1 = fba_bin<KMAX>(b, K, p);
      reinterpret_cast<float4*>(out)[i] = make_float4(r0.x, r0.y, r1.x, r1.y);
    } else {
      out[i] = fba_bin<KMAX>(a, K, p);
    }
  }
}
template <int KMAX>
static void fba_launch(const PtrPack& pk, int K, float p, float2* out, long long n, bool vec, cudaStream_t stream) {
  if (vec)
    fba_combine_kernel<KMAX, 2><<<grid_for(n / 2, 256, 8), 256, 0, stream>>>(pk, K, p, out, n);
  else
    fba_combine_kernel<KMAX, 1><<<grid_for(n, 256, 8), 256, 0, stream>>>(pk, K, p, out, n);
}
// VT = float4 (element count a multiple of 4, 16-byte aligned bases) or float; same sum order and the same division as the statement.
__device__ __forceinline__ void mean_add(float& s, const float& v) { s += v; }
__device__ __forceinline__ void mean_add(float4& s, const float4& v) {
  s.x += v.x;
  s.y += v.y;
  s.z += v.z;
  s.w += v.w;
}
__device__ __forceinline__ float mean_div(const float& s, float k) { return s / k; }
__device__ __forceinline__ float4 mean_div(const float4& s, float k) { return make_float4(s.x / k, s.y / k, s.z / k, s.w / k); }
template <typename VT, int KMAX>
__global__ void __launch_bounds__(256) mean_stack_kernel(PtrPack vp, int K, VT* out, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    VT v[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k)  // all K loads in flight (static indices: the pointer pack stays in the parameter bank)
      if (k < K) v[k] = reinterpret_cast<const VT*>(vp.p[k])[i];
    VT s = v[0];
#pragma unroll
    for (int k = 1; k < KMAX; ++k)
      if (k < K) mean_add(s, v[k]);
    out[i] = mean_div(s, (float)K);
  }
}
template <int KMAX>
static void mean_launch(const PtrPack& pk, int K, float* out, long long n, bool vec, cudaStream_t stream) {
  if (vec)
    mean_stack_kernel<float4, KMAX><<<grid_for(n / 4, 256, 8), 256, 0, stream>>>(pk, K, reinterpret_cast<float4*>(out), n / 4);
  else
    mean_stack_kernel<float, KMAX><<<grid_for(n, 256, 8), 256, 0, stream>>>(pk, K, out, n);
}

// =================================================================================================
// Activation backward from the activation OUTPUT: dy = da * (a > 0 ? 1 : slope)   (slope = 0 for ReLU)
// =================================================================================================
__global__ void __launch_bounds__(256) act_bwd_kernel(const __nv_bfloat16* a, long long lda, const __nv_bfloat16* da,
                                                      long long ldda, __nv_bfloat16* dy, long long lddy, long long vox,
                                                      int C, float slope) {
  const int groups = C / 8;
  const long long items = vox * groups;
  for (long long it = blockIdx.x * (long long)blockDim.x + threadIdx.x; it < items; it += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(it % groups);
    const long long v = it / groups;
    float fa[8], fd[8], o[8];
    bf16x8_to_float(*reinterpret_cast<const uint4*>(a + v * lda + g * 8), fa);
    bf16x8_to_float(*reinterpret_cast<const uint4*>(da + v * ldda + g * 8), fd);
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = fa[i] > 0.f ? fd[i] : fd[i] * slope;
    *reinterpret_cast<uint4*>(dy + v * lddy + g * 8) = float_to_bf16x8(o);
  }
}

}  // namespace rehr

// =================================================================================================
// C-ABI
// =================================================================================================
using namespace rehr;

extern "C" {

int rehr_instnorm_stats_tiles(const rehr_tensor* x) { return x ? stat_tiles(x) : 0; }

int rehr_instnorm_stats(const rehr_tensor* x, float* partial, rehr_stream stream) {
  if (!bf16_tensor_ok(x) || !partial) return REHR_BAD_SHAPE;
  StatArgs a{};
  a.y = reinterpret_cast<const __nv_bfloat16*>(x->ptr);
  a.y_f16 = x->dtype == REHR_F16;
  a.ld_y = x->ld;
  a.partial = partial;
  a.V = voxels_per_sample(x);
  a.C = x->c;
  a.tiles = stat_tiles(x);
  a.vpb = stat_vox_per_block(x);
  return launch_in_reduce<0>(a, x->n, (cudaStream_t)stream);
}

int rehr_instnorm_finalize(const float* partial, int n, int tiles, int c, long long count, float eps, float* mean,
                           float* rstd, rehr_stream stream) {
  if (!partial || !mean || !rstd || count <= 0) return REHR_BAD_SHAPE;
  if (tiles >= 256)
    in_finalize_kernel<8><<<dim3((c + 7) / 8, n), 32 * kFinLanes, 0, (cudaStream_t)stream>>>(partial, n, tiles, c, 1.0 / (double)count, eps, mean,
                                                                            rstd);
  else
    in_finalize_kernel<32><<<dim3((c + 31) / 32, n), 32 * kFinLanes, 0, (cudaStream_t)stream>>>(partial, n, tiles, c, 1.0 / (double)count, eps, mean,
                                                                              rstd);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_instnorm_lrelu_apply(const rehr_tensor* y, const float* mean, const float* rstd, const float* gamma,
                              const float* beta, float slope, const rehr_tensor* a, const rehr_tensor* a2, rehr_stream stream) {
  if (!bf16_tensor_ok(y) || !bf16_tensor_ok(a) || y->c != a->c || y->n != a->n || voxels_per_sample(y) != voxels_per_sample(a))
    return REHR_BAD_SHAPE;
  if (a2 && (!bf16_tensor_ok(a2) || a2->c != y->c || a2->n != y->n || voxels_per_sample(a2) != voxels_per_sample(y))) return REHR_BAD_SHAPE;
  ApplyArgs p{};
  p.y = reinterpret_cast<const __nv_bfloat16*>(y->ptr);
  p.out = reinterpret_cast<__nv_bfloat16*>(a->ptr);
  p.y_f16 = y->dtype == REHR_F16;
  p.out_f16 = a->dtype == REHR_F16;
  p.range = range_target(p.out_f16 || (a2 && a2->dtype == REHR_F16));
  if (a2) {
    p.out2 = reinterpret_cast<__nv_bfloat16*>(a2->ptr);
    p.ld_o2 = a2->ld;
    p.out2_f16 = a2->dtype == REHR_F16;
  }
  p.ld_y = y->ld;
  p.ld_o = a->ld;
  p.mean = mean;
  p.rstd = rstd;
  p.gamma = gamma;
  p.beta = beta;
  p.slope = slope;
  p.V = voxels_per_sample(y);
  p.C = y->c;
  return launch_in_apply<0>(p, y->n, (cudaStream_t)stream);
}

int rehr_instnorm_lrelu_bwd_reduce(const rehr_tensor* y, const rehr_tensor* da1, const rehr_tensor* da2, const float* mean,
                                   const float* rstd, const float* gamma, const float* beta, float slope, float* partial,
                                   rehr_stream stream) {
  if (!bf16_tensor_ok(y) || !bf16_tensor_ok(da1) || (da2 && !bf16_tensor_ok(da2)) || !partial) return REHR_BAD_SHAPE;
  StatArgs a{};
  a.y = reinterpret_cast<const __nv_bfloat16*>(y->ptr);
  a.y_f16 = y->dtype == REHR_F16;
  a.da1 = reinterpret_cast<const __nv_bfloat16*>(da1->ptr);
  a.da2 = da2 ? reinterpret_cast<const __nv_bfloat16*>(da2->ptr) : nullptr;
  a.ld_y = y->ld;
  a.ld_a1 = da1->ld;
  a.ld_a2 = da2 ? da2->ld : 0;
  a.mean = mean;
  a.rstd = rstd;
  a.gamma = gamma;
  a.beta = beta;
  a.slope = slope;
  a.partial = partial;
  a.V = voxels_per_sample(y);
  a.C = y->c;
  a.tiles = stat_tiles(y);
  a.vpb = stat_vox_per_block(y);
  return launch_in_reduce<1>(a, y->n, (cudaStream_t)stream);
}

int rehr_instnorm_lrelu_bwd_finalize(const float* partial, int n, int tiles, int c, const float* rstd, float* sums,
                                     float* dgamma, float* dbeta, int accumulate, rehr_stream stream) {
  (void)rstd;
  if (!partial || !sums) return REHR_BAD_SHAPE;
  in_bwd_finalize_kernel<<<(c + 31) / 32, 32 * kFinLanes, 0, (cudaStream_t)stream>>>(partial, n, tiles, c, sums, dgamma, dbeta, accumulate);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_instnorm_lrelu_bwd_apply(const rehr_tensor* y, const rehr_tensor* da1, const rehr_tensor* da2, const float* mean,
                                  const float* rstd, const float* gamma, const float* beta, float slope, const float* sums,
                                  const rehr_tensor* dy, rehr_stream stream) {
  if (!bf16_tensor_ok(y) || !bf16_tensor_ok(da1) || (da2 && !bf16_tensor_ok(da2)) || !bf16_tensor_ok(dy) || !sums)
    return REHR_BAD_SHAPE;
  ApplyArgs p{};
  p.y = reinterpret_cast<const __nv_bfloat16*>(y->ptr);
  p.y_f16 = y->dtype == REHR_F16;
  p.out_f16 = dy->dtype == REHR_F16;
  p.da1 = reinterpret_cast<const __nv_bfloat16*>(da1->ptr);
  p.da2 = da2 ? reinterpret_cast<const __nv_bfloat16*>(da2->ptr) : nullptr;
  p.out = reinterpret_cast<__nv_bfloat16*>(dy->ptr);
  p.ld_y = y->ld;
  p.ld_a1 = da1->ld;
  p.ld_a2 = da2 ? da2->ld : 0;
  p.ld_o = dy->ld;
  p.mean = mean;
  p.rstd = rstd;
  p.gamma = gamma;
  p.beta = beta;
  p.sums = sums;
  p.slope = slope;
  p.V = voxels_per_sample(y);
  p.C = y->c;
  return launch_in_apply<1>(p, y->n, (cudaStream_t)stream);
}

int rehr_pointwise_fwd(const rehr_tensor* x, const float* w, const float* bias, float* y_ncdhw, int cout, rehr_stream stream) {
  if (!bf16_tensor_ok(x) || !w || !y_ncdhw) return REHR_BAD_SHAPE;
  if (cout > kPwCoutLimit || x->c > kPwMaxCin) return REHR_UNSUPPORTED;
  const long long V = voxels_per_sample(x);
  const dim3 grid((unsigned)std::max(1, grid_for(V, 256, 8)), (unsigned)x->n);
  const __nv_bfloat16* xp = reinterpret_cast<const __nv_bfloat16*>(x->ptr);
  const int xf = x->dtype == REHR_F16;
  if (cout <= 2 && x->c == 32)  // the nnU-Net segmentation head (decoder.seg_layers[-1], models/seg_model.py:44)
    pointwise_fwd_kernel<2, 32><<<grid, 256, 0, (cudaStream_t)stream>>>(xp, x->ld, w, bias, y_ncdhw, V, x->c, cout, xf);
  else if (cout <= 2)
    pointwise_fwd_kernel<2, 0><<<grid, 256, 0, (cudaStream_t)stream>>>(xp, x->ld, w, bias, y_ncdhw, V, x->c, cout, xf);
  else if (cout <= 4)
    pointwise_fwd_kernel<4, 0><<<grid, 256, 0, (cudaStream_t)stream>>>(xp, x->ld, w, bias, y_ncdhw, V, x->c, cout, xf);
  else
    pointwise_fwd_kernel<8, 0><<<grid, 256, 0, (cudaStream_t)stream>>>(xp, x->ld, w, bias, y_ncdhw, V, x->c, cout, xf);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

size_t rehr_pointwise_bwd_workspace(const rehr_tensor* x, int cout) {
  if (!x) return 0;
  return (size_t)pointwise_bwd_blocks(x) * x->n * cout * (x->c + 1) * sizeof(float);
}

int rehr_pointwise_bwd(const rehr_tensor* x, const float* dy_ncdhw, const float* w, int cout, const rehr_tensor* dx, float* dw,
                       float* dbias, int accumulate, void* ws, size_t ws_bytes, rehr_stream stream) {
  if (!bf16_tensor_ok(x) || !dy_ncdhw || !w || (dx && !bf16_tensor_ok(dx))) return REHR_BAD_SHAPE;
  if (cout > kPwCoutLimit || x->c > kPwMaxCin) return REHR_UNSUPPORTED;
  if (ws_bytes < rehr_pointwise_bwd_workspace(x, cout) || !ws) return REHR_WORKSPACE;
  const long long V = voxels_per_sample(x);
  const int bx = pointwise_bwd_blocks(x);
  const int blocks = bx * x->n;
  const dim3 grid((unsigned)bx, (unsigned)x->n);
  const __nv_bfloat16* xp = reinterpret_cast<const __nv_bfloat16*>(x->ptr);
  __nv_bfloat16* dxp = dx ? reinterpret_cast<__nv_bfloat16*>(dx->ptr) : nullptr;
  const long long lddx = dx ? dx->ld : 0;
  float* wsp = reinterpret_cast<float*>(ws);
  const int xf = x->dtype == REHR_F16;
  if (dx && dx->dtype != REHR_BF16) return REHR_UNSUPPORTED;  // gradients are bf16
  if (cout <= 2)
    pointwise_bwd_kernel<2><<<grid, 256, 0, (cudaStream_t)stream>>>(xp, x->ld, dy_ncdhw, w, dxp, lddx, wsp, V, x->c, cout, xf);
  else if (cout <= 4)
    pointwise_bwd_kernel<4><<<grid, 256, 0, (cudaStream_t)stream>>>(xp, x->ld, dy_ncdhw, w, dxp, lddx, wsp, V, x->c, cout, xf);
  else
    pointwise_bwd_kernel<8><<<grid, 256, 0, (cudaStream_t)stream>>>(xp, x->ld, dy_ncdhw, w, dxp, lddx, wsp, V, x->c, cout, xf);
  REHR_CHECK_LAUNCH();
  const int outs = cout * (x->c + 1);
  pointwise_bwd_reduce_kernel<<<outs, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float*>(ws), blocks, x->c, cout, dw,
                                                                     dbias, accumulate);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

size_t rehr_channel_sum_workspace(const rehr_tensor* x) {
  if (!x) return 0;
  return (size_t)channel_sum_blocks(x) * x->c * sizeof(float);
}
int rehr_channel_sum(const rehr_tensor* x, float* out, int accumulate, void* ws, size_t ws_bytes, rehr_stream stream) {
  if (!bf16_tensor_ok(x) || !out) return REHR_BAD_SHAPE;
  if (ws_bytes < rehr_channel_sum_workspace(x) || !ws) return REHR_WORKSPACE;
  const int blocks = channel_sum_blocks(x);
  channel_sum_kernel<<<blocks, 256, x->c * sizeof(float), (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(x->ptr), x->ld, (long long)x->n * voxels_per_sample(x), x->c, reinterpret_cast<float*>(ws));
  REHR_CHECK_LAUNCH();
  channel_sum_reduce_kernel<<<(x->c + 31) / 32, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float*>(ws), blocks, x->c, out,
                                                                             accumulate);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_upsample_linear_d(const rehr_tensor* x, const rehr_tensor* y, rehr_stream stream) {
  if (!bf16_tensor_ok(x) || !bf16_tensor_ok(y) || x->c != y->c || x->n != y->n || x->h != y->h || x->w != y->w) return REHR_BAD_SHAPE;
  const long long HW = (long long)x->h * x->w;
  if (y->d >= x->d) {
    const long long items = (long long)x->n * x->d * HW * (x->c / 8);
    upsample_d_src_kernel<<<grid_for(items, 256, 8), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const __nv_bfloat16*>(x->ptr), x->ld, reinterpret_cast<__nv_bfloat16*>(y->ptr), y->ld, x->n, x->d, y->d, HW, x->c,
        x->dtype == REHR_F16, y->dtype == REHR_F16, range_target(y->dtype == REHR_F16));
    REHR_CHECK_LAUNCH();
    return REHR_OK;
  }
  const long long items = (long long)y->n * y->d * HW * (y->c / 8);
  upsample_d_kernel<<<grid_for(items, 256, 8), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __nv_bfloat16*>(x->ptr), x->ld,
                                                                           reinterpret_cast<__nv_bfloat16*>(y->ptr), y->ld, x->n, x->d,
                                                                           y->d, HW, x->c, x->dtype == REHR_F16, y->dtype == REHR_F16,
                                                                           range_target(y->dtype == REHR_F16));
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}
int rehr_upsample_linear_d_bwd(const rehr_tensor* dy, const rehr_tensor* dx, rehr_stream stream) {
  if (!bf16_tensor_ok(dx) || !bf16_tensor_ok(dy) || dx->c != dy->c || dx->n != dy->n || dx->h != dy->h || dx->w != dy->w)
    return REHR_BAD_SHAPE;
  const long long HW = (long long)dx->h * dx->w;
  const long long items = (long long)dx->n * dx->d * HW * (dx->c / 8);
  upsample_d_bwd_kernel<<<grid_for(items, 256, 8), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __nv_bfloat16*>(dy->ptr),
                                                                               dy->ld, reinterpret_cast<__nv_bfloat16*>(dx->ptr),
                                                                               dx->ld, dx->n, dx->d, dy->d, HW, dx->c);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_ncdhw_f32_to_ndhwc_bf16(const float* src, const rehr_tensor* dst, rehr_stream stream) {
  if (!src || !dst || !dst->ptr) return REHR_BAD_SHAPE;
  const long long V = voxels_per_sample(dst);
  dim3 grid((unsigned)((V + 31) / 32), (unsigned)((dst->c + 31) / 32), (unsigned)dst->n);
  ncdhw_to_ndhwc_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, reinterpret_cast<__nv_bfloat16*>(dst->ptr), dst->ld, V, dst->c);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}
int rehr_ndhwc_bf16_to_ncdhw_f32(const rehr_tensor* src, float* dst, rehr_stream stream) {
  if (!src || !dst || !src->ptr) return REHR_BAD_SHAPE;
  const long long V = voxels_per_sample(src);
  dim3 grid((unsigned)((V + 31) / 32), (unsigned)((src->c + 31) / 32), (unsigned)src->n);
  ndhwc_to_ncdhw_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const unsigned short*>(src->ptr), src->ld, dst, V, src->c,
                                                                src->dtype == REHR_F16);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_convert16(const rehr_tensor* src, const rehr_tensor* dst, rehr_stream stream) {
  if (!bf16_tensor_ok(src) || !bf16_tensor_ok(dst) || src->c != dst->c || src->n != dst->n || voxels_per_sample(src) != voxels_per_sample(dst))
    return REHR_BAD_SHAPE;
  const long long vox = (long long)src->n * voxels_per_sample(src);
  convert16_kernel<<<grid_for(vox * (src->c / 8), 256, 8), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(src->ptr), src->ld, src->dtype == REHR_F16, reinterpret_cast<__nv_bfloat16*>(dst->ptr), dst->ld,
      dst->dtype == REHR_F16, vox, src->c, range_target(dst->dtype == REHR_F16));
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_segate_scale_add_act(const rehr_tensor* x, const float* gate, const rehr_tensor* residual, int act, float slope,
                              const rehr_tensor* y, rehr_stream stream) {
  if (!bf16_tensor_ok(x) || !bf16_tensor_ok(y) || (residual && !bf16_tensor_ok(residual)) || x->c != y->c) return REHR_BAD_SHAPE;
  const long long V = voxels_per_sample(x);
  const long long items = (long long)x->n * V * (x->c / 8);
  segate_kernel<<<grid_for(items, 256, 8), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(x->ptr), x->ld, gate, residual ? reinterpret_cast<const __nv_bfloat16*>(residual->ptr) : nullptr,
      residual ? residual->ld : 0, reinterpret_cast<__nv_bfloat16*>(y->ptr), y->ld, x->n, V, x->c, act, slope);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

// d(gate) partial sums: partial [n][rehr_instnorm_stats_tiles(x)][c][2] (second slot zero), reduce with
// rehr_instnorm_lrelu_bwd_finalize (sums[n][c][0] = d gate).
int rehr_segate_bwd_reduce(const rehr_tensor* x, const rehr_tensor* y, const rehr_tensor* dy, int act, float slope, float* partial,
                           rehr_stream stream) {
  if (!bf16_tensor_ok(x) || !bf16_tensor_ok(dy) || (act != REHR_ACT_NONE && !bf16_tensor_ok(y)) || !partial) return REHR_BAD_SHAPE;
  const int groups = x->c / 8;
  if (groups > kStatThreads) return REHR_UNSUPPORTED;
  const int lanes = kStatThreads / groups;
  const int tiles = stat_tiles(x), vpb = stat_vox_per_block(x);
  const size_t smem = (size_t)lanes * x->c * sizeof(float);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(segate_bwd_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      g_last_cuda_error = (int)e;
      return REHR_CUDA_ERROR;
    }
  }
  dim3 grid(tiles, x->n);
  segate_bwd_kernel<0><<<grid, kStatThreads, smem, (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(x->ptr), x->ld, y ? reinterpret_cast<const __nv_bfloat16*>(y->ptr) : nullptr, y ? y->ld : 0,
      reinterpret_cast<const __nv_bfloat16*>(dy->ptr), dy->ld, nullptr, nullptr, nullptr, 0, nullptr, 0, partial, voxels_per_sample(x),
      x->c, tiles, vpb, act, slope);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

// dx = dy*act'(y)*gate[n,c] + shift[n,c];  dres (optional) = dy*act'(y)
int rehr_segate_bwd_apply(const rehr_tensor* y, const rehr_tensor* dy, int act, float slope, const float* gate, const float* shift,
                          const rehr_tensor* dx, const rehr_tensor* dres, rehr_stream stream) {
  if (!bf16_tensor_ok(dy) || !bf16_tensor_ok(dx) || (act != REHR_ACT_NONE && !bf16_tensor_ok(y)) || (dres && !bf16_tensor_ok(dres)))
    return REHR_BAD_SHAPE;
  const int groups = dy->c / 8;
  if (groups > kStatThreads) return REHR_UNSUPPORTED;
  const int tiles = stat_tiles(dy), vpb = stat_vox_per_block(dy);
  dim3 grid(tiles, dy->n);
  segate_bwd_kernel<1><<<grid, kStatThreads, 0, (cudaStream_t)stream>>>(
      nullptr, 0, y ? reinterpret_cast<const __nv_bfloat16*>(y->ptr) : nullptr, y ? y->ld : 0,
      reinterpret_cast<const __nv_bfloat16*>(dy->ptr), dy->ld, gate, shift, reinterpret_cast<__nv_bfloat16*>(dx->ptr), dx->ld,
      dres ? reinterpret_cast<__nv_bfloat16*>(dres->ptr) : nullptr, dres ? dres->ld : 0, nullptr, voxels_per_sample(dy), dy->c, tiles, vpb,
      act, slope);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_sw_accumulate(void* logits_f16, void* npred_f16, const void* pred, int pred_is_f32, const void* gauss_f16, int C, int VD,
                       int VH, int VW, int TD, int TH, int TW, int od, int oh, int ow, rehr_stream stream) {
  if (!logits_f16 || !pred) return REHR_BAD_SHAPE;  // npred_f16 may be NULL: blend the logits only
  if (od < 0 || oh < 0 || ow < 0 || od + TD > VD || oh + TH > VH || ow + TW > VW) return REHR_BAD_SHAPE;
  const long long tv = (long long)TD * TH * TW;
  const uintptr_t bases = reinterpret_cast<uintptr_t>(logits_f16) | reinterpret_cast<uintptr_t>(npred_f16) |
                          reinterpret_cast<uintptr_t>(pred) | reinterpret_cast<uintptr_t>(gauss_f16);  // NULL contributes nothing
  if (TW % 8 == 0 && VW % 8 == 0 && ow % 8 == 0 && (bases & 15) == 0 && tv > 0) {
    sw_accumulate_vec8_kernel<<<grid_for(tv / 8, 256, 8), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<__half*>(logits_f16), reinterpret_cast<__half*>(npred_f16), pred, pred_is_f32,
        reinterpret_cast<const __half*>(gauss_f16), C, VD, VH, VW, TD, TH, TW, od, oh, ow);
    REHR_CHECK_LAUNCH();
    return REHR_OK;
  }
  sw_accumulate_kernel<<<grid_for(tv, 256, 8), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<__half*>(logits_f16), reinterpret_cast<__half*>(npred_f16), pred, pred_is_f32,
      reinterpret_cast<const __half*>(gauss_f16), C, VD, VH, VW, TD, TH, TW, od, oh, ow);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}
int rehr_sw_finalize(void* logits_f16, const void* npred_f16, int C, long long voxels, int* inf_flag, rehr_stream stream) {
  if (!logits_f16 || !npred_f16) return REHR_BAD_SHAPE;
  if (voxels % 8 == 0 && voxels > 0 && ((reinterpret_cast<uintptr_t>(logits_f16) | reinterpret_cast<uintptr_t>(npred_f16)) & 15) == 0) {
    sw_finalize_vec8_kernel<<<grid_for(voxels / 8, 256, 8), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<__half*>(logits_f16), reinterpret_cast<const __half*>(npred_f16), C, voxels, inf_flag);
    REHR_CHECK_LAUNCH();
    return REHR_OK;
  }
  sw_finalize_kernel<<<grid_for(voxels, 256, 8), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<__half*>(logits_f16),
                                                                             reinterpret_cast<const __half*>(npred_f16), C, voxels,
                                                                             inf_flag);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_blur1d(const float* x, const float* taps, int L, float* y, long long Z, int X, int Y, rehr_stream stream) {
  if (!x || !taps || !y || L <= 0) return REHR_BAD_SHAPE;
  if (L > kBlurMaxTaps) return REHR_UNSUPPORTED;
  const size_t smem = (size_t)(kBlurRows + L - 1) * 128 * sizeof(float);
  if (smem > 48 * 1024) REHR_SET_MAX_SMEM_ONCE(blur1d_kernel, (kBlurRows + kBlurMaxTaps) * 128 * sizeof(float));
  const long long tiles = Z * (long long)((X + kBlurRows - 1) / kBlurRows) * ((Y + 127) / 128);
  const int grid = (int)std::max<long long>(1, std::min<long long>(tiles, (long long)sm_count() * 6));
  const bool vec = Y % 4 == 0 && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0;
  if (vec) {
    if (smem > 48 * 1024) REHR_SET_MAX_SMEM_ONCE(blur1d_vec4_kernel, (kBlurRows + kBlurMaxTaps) * 128 * sizeof(float));
    blur1d_vec4_kernel<<<grid, 128, smem, (cudaStream_t)stream>>>(x, y, taps, L, Z, X, Y);
  } else {
    blur1d_kernel<<<grid, 128, smem, (cudaStream_t)stream>>>(x, y, taps, L, Z, X, Y);
  }
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

static int uasr_blocks(long long total) { return (int)std::max<long long>(1, std::min<long long>((total + 127) / 128, (long long)sm_count() * 16)); }

int rehr_uasr_mixture_blocks(long long pixels, int n_out) { return uasr_blocks(pixels * n_out); }

int rehr_uasr_mixture_fwd(const float* out_cl, const float* ue_cl, const float* w, const float* b, float* res, float* unc, long long batch,
                          long long hw, int n_out, int experts, rehr_stream stream) {
  if (!out_cl || !ue_cl || !w || !b || !res || !unc || batch <= 0 || hw <= 0 || n_out <= 0) return REHR_BAD_SHAPE;
  if (experts != kUasrE) return REHR_UNSUPPORTED;
  if (((reinterpret_cast<uintptr_t>(out_cl) | reinterpret_cast<uintptr_t>(ue_cl)) & 15) != 0) return REHR_BAD_ALIGNMENT;
  UasrArgs a{};
  a.out = out_cl; a.ue = ue_cl; a.w = w; a.b = b; a.res = res; a.unc = unc;
  a.pixels = batch * hw; a.HW = hw; a.n_out = n_out;
  uasr_mixture_fwd_kernel<<<uasr_blocks(a.pixels * n_out), 128, 0, (cudaStream_t)stream>>>(a);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_uasr_mixture_bwd(const float* out_cl, const float* ue_cl, const float* w, const float* b, const float* d_res, const float* d_unc,
                          float* d_out_cl, float* d_ue_cl, float* partial, long long batch, long long hw, int n_out, int experts,
                          rehr_stream stream) {
  if (!out_cl || !ue_cl || !w || !b || !d_out_cl || !d_ue_cl || !partial || batch <= 0 || hw <= 0 || n_out <= 0) return REHR_BAD_SHAPE;
  if (experts != kUasrE) return REHR_UNSUPPORTED;
  UasrArgs a{};
  a.out = out_cl; a.ue = ue_cl; a.w = w; a.b = b; a.d_res = d_res; a.d_unc = d_unc; a.d_out = d_out_cl; a.d_ue = d_ue_cl; a.partial = partial;
  a.pixels = batch * hw; a.HW = hw; a.n_out = n_out;
  uasr_mixture_bwd_kernel<<<uasr_blocks(a.pixels * n_out), 128, 0, (cudaStream_t)stream>>>(a);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_bspline_prefilter_axis(float* c, long long outer, int n, long long inner, rehr_stream stream) {
  if (!c || outer <= 0 || n <= 0 || inner <= 0) return REHR_BAD_SHAPE;
  if (n < 2) return REHR_OK;
  const long long lines = outer * inner;
  bspline_prefilter_kernel<<<(unsigned)((lines + 127) / 128), 128, 0, (cudaStream_t)stream>>>(c, outer, n, inner);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_affine_sample2d(const float* src, float* dst, const float* affine, int slices, int x, int y, int px, int py, int slices_per_sample,
                         int order, float cval, const float* labels_host, int n_labels, rehr_stream stream) {
  if (!src || !dst || !affine || slices <= 0 || x <= 0 || y <= 0 || px <= 0 || py <= 0 || slices_per_sample <= 0) return REHR_BAD_SHAPE;
  if (order != 3 && order != 1) return REHR_UNSUPPORTED;
  if (order == 1 && (n_labels <= 0 || n_labels > 8 || !labels_host)) return REHR_UNSUPPORTED;
  AffineSampleArgs a{};
  a.src = src; a.dst = dst; a.affine = affine;
  a.S = slices; a.X = x; a.Y = y; a.PX = px; a.PY = py; a.per_sample = slices_per_sample;
  a.order = order; a.cval = cval; a.n_labels = order == 1 ? n_labels : 0;
  for (int i = 0; i < a.n_labels; ++i) a.labels[i] = labels_host[i];
  const long long total = (long long)slices * px * py;
  const int grid = (int)std::max<long long>(1, std::min<long long>((total + 255) / 256, (long long)sm_count() * 16));
  affine_sample2d_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_resample_axis(const float* x, float* y, long long outer, int n_in, int n_out, long long inner, float step, int order,
                       rehr_stream stream) {
  if (!x || !y || outer <= 0 || n_in <= 0 || n_out <= 0 || inner <= 0 || !(step > 0.f)) return REHR_BAD_SHAPE;
  if (order != 0 && order != 3) return REHR_UNSUPPORTED;
  const long long total = outer * n_out * inner;
  const int grid = (int)std::max<long long>(1, std::min<long long>((total + 255) / 256, (long long)sm_count() * 16));
  resample_axis_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, outer, n_in, n_out, inner, step, order);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_rot90(const void* src, void* dst, int X, int Y, long long inner_bytes, int k, rehr_stream stream) {
  if (!src || !dst || X <= 0 || Y <= 0 || inner_bytes <= 0) return REHR_BAD_SHAPE;
  k = ((k % 4) + 4) % 4;
  const long long total_bytes = (long long)X * Y * inner_bytes;
  if (k == 0) {
    cudaError_t e = cudaMemcpyAsync(dst, src, (size_t)total_bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    if (e != cudaSuccess) {
      g_last_cuda_error = (int)e;
      return REHR_CUDA_ERROR;
    }
    return REHR_OK;
  }
  const bool a16 = inner_bytes % 16 == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0;
  const bool a4 = inner_bytes % 4 == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 3) == 0;
  if (a16) {
    const long long inner = inner_bytes / 16;
    rot90_kernel<uint4><<<grid_for((long long)X * Y * inner, 256, 8), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint4*>(src), reinterpret_cast<uint4*>(dst), X, Y, inner, k);
  } else if (a4) {
    const long long inner = inner_bytes / 4;
    rot90_kernel<uint32_t><<<grid_for((long long)X * Y * inner, 256, 8), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint32_t*>(src), reinterpret_cast<uint32_t*>(dst), X, Y, inner, k);
  } else {
    rot90_kernel<uint8_t><<<grid_for(total_bytes, 256, 8), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const uint8_t*>(src), reinterpret_cast<uint8_t*>(dst), X, Y, inner_bytes, k);
  }
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_fba_combine(const void* const* spectra, int K, float p, void* out, long long n, rehr_stream stream) {
  if (!spectra || !out || K <= 0) return REHR_BAD_SHAPE;
  if (K > kMaxFuse) return REHR_UNSUPPORTED;
  PtrPack pk{};
  for (int i = 0; i < K; ++i) pk.p[i] = spectra[i];
  uintptr_t bases = reinterpret_cast<uintptr_t>(out);
  for (int i = 0; i < K; ++i) bases |= reinterpret_cast<uintptr_t>(spectra[i]);
  const bool vec = n % 2 == 0 && (bases & 15) == 0;
  if (K <= 4)
    fba_launch<4>(pk, K, p, reinterpret_cast<float2*>(out), n, vec, (cudaStream_t)stream);
  else if (K <= 8)
    fba_launch<8>(pk, K, p, reinterpret_cast<float2*>(out), n, vec, (cudaStream_t)stream);
  else
    fba_launch<16>(pk, K, p, reinterpret_cast<float2*>(out), n, vec, (cudaStream_t)stream);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}
int rehr_mean_stack(const float* const* vols, int K, float* out, long long n, rehr_stream stream) {
  if (!vols || !out || K <= 0) return REHR_BAD_SHAPE;
  if (K > kMaxFuse) return REHR_UNSUPPORTED;
  PtrPack pk{};
  for (int i = 0; i < K; ++i) pk.p[i] = vols[i];
  uintptr_t bases = reinterpret_cast<uintptr_t>(out);
  for (int i = 0; i < K; ++i) bases |= reinterpret_cast<uintptr_t>(vols[i]);
  const bool vec = n % 4 == 0 && (bases & 15) == 0;
  if (K <= 4)
    mean_launch<4>(pk, K, out, n, vec, (cudaStream_t)stream);
  else if (K <= 8)
    mean_launch<8>(pk, K, out, n, vec, (cudaStream_t)stream);
  else
    mean_launch<16>(pk, K, out, n, vec, (cudaStream_t)stream);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_act_bwd(const rehr_tensor* a, const rehr_tensor* da, int act, float slope, const rehr_tensor* dy, rehr_stream stream) {
  if (!bf16_tensor_ok(a) || !bf16_tensor_ok(da) || !bf16_tensor_ok(dy)) return REHR_BAD_ALIGNMENT;
  if (a->c != da->c || a->c != dy->c) return REHR_BAD_SHAPE;
  if (act != REHR_ACT_RELU && act != REHR_ACT_LRELU) return REHR_UNSUPPORTED;
  const long long vox = (long long)a->n * voxels_per_sample(a);
  act_bwd_kernel<<<grid_for(vox * (a->c / 8), 256, 8), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(a->ptr), a->ld, reinterpret_cast<const __nv_bfloat16*>(da->ptr), da->ld,
      reinterpret_cast<__nv_bfloat16*>(dy->ptr), dy->ld, vox, a->c, act == REHR_ACT_RELU ? 0.f : slope);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

}  // extern "C"
