// Tensor-core stem for the 1-channel nnU-Net input conv (k = 3x3x3, stride 1, pad 1, Cin = 1, Cout = 32; built at
// models/seg_model.py:174-191 with the plan of train_all.py:474-493): forward and weight gradient.
//
// With one input channel the contraction length is the 27 taps, so there is nothing for TMA / tcgen05 to stream: the operand is
// an im2col of a tiny fp32 halo tile that has to be gathered by threads anyway.  The CUDA-core versions (smallcin.cu) spend
// 9 shared loads per 32 FMAs and run at ~22 TFLOP/s (0.33 ms forward, 0.46 ms weight gradient on 2x128^3); both layers are
// bound by ONE pass over the 268 MB bf16 activation (~45 us).  Here the gather feeds warp-level mma.sync.m16n8k16 (bf16 inputs,
// fp32 accumulation) -- 16 voxels x 32 channels per 8 MMAs -- and the fp32 image / weights are split into bf16 hi + lo parts
// (three MMAs for hi*hi + lo*hi + hi*lo in the forward, two in the weight gradient where dY is exactly bf16), so the result
// keeps the fp32 accuracy of the CUDA-core path it replaces (the stem sees the caller's fp32 image, train_all.py:524).
//
//   forward : Y[v][co]      = sum_tap  Xcol[v][tap] * W[co][tap]        M = 16 voxels of a row, N = 32, K = 27 (padded to 32)
//   wgrad   : dW^T[tap][co] = sum_v    Xcol[v][tap] * dY[v][co]         M = 32 taps,           N = 32, K = voxels
//
// A CTA (8 warps) stages the 3 x 10 x (W + halo) fp32 input rows that 8 output rows need; warp = output row.
#include "engine.h"
#include "ptx.cuh"

#include <algorithm>
#include <cstdint>

namespace rehr {

struct StemArgs {
  const float* x;       // [n][1][d][h][w] fp32
  const float* w;       // [32][27] fp32
  const float* bias;    // [32] or null
  __nv_bfloat16* y;     // NDHWC bf16 (forward output / weight-gradient dY)
  long long ldy;        // voxel pitch of y in elements
  float* ws;            // wgrad: per-CTA partials [cta][27][32]
  int n, d, h, wd;
  int act;
  float slope;
  int planar;           // 1: k = (1,3,3), pad (0,1,1) (the stem of anisotropic plans): 9 taps, one staged plane
  int y_f16;            // forward: storage format of y (rehr_dtype); the weight gradient's dY is always bf16
  RangeSlot* range;     // forward: fp16 saturation record of y (rehr_range_sink), null = not checked
};

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// (v0, v1) -> packed bf16 hi parts and packed bf16 residuals (v - hi)
__device__ __forceinline__ void split_bf16x2(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 h0 = __float2bfloat16(v0), h1 = __float2bfloat16(v1);
  const float r0 = v0 - __bfloat162float(h0), r1 = v1 - __bfloat162float(h1);
  hi = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
  lo = pack_bf16x2(r0, r1);
}

static constexpr int kStemRowPad = 80;  // bytes per staged 32-channel bf16 voxel row (64 + 16: conflict-free 4 B / 16 B access)

// stage the rows oz-1..oz+1 x oy0-1..oy0+8 of sample nn, columns -1 .. Wp (zero outside the volume); Wa = Wp + 2
__device__ __forceinline__ void stem_stage_rows(const StemArgs& a, float* sx, int Wa, int nn, int oz, int oy0) {
  const long long in_plane = (long long)a.h * a.wd, in_vol = in_plane * a.d;
  const int rows = a.planar ? 10 : 30;
  for (int i = threadIdx.x; i < rows * Wa; i += blockDim.x) {
    const int xx = i % Wa;
    const int q = i / Wa;
    const int yy = q % 10, kz = q / 10;
    const int iz = a.planar ? oz : oz + kz - 1, iy = oy0 + yy - 1, ix = xx - 1;
    float v = 0.f;
    if (iz >= 0 && iz < a.d && iy >= 0 && iy < a.h && ix >= 0 && ix < a.wd)
      v = __ldg(a.x + (long long)nn * in_vol + iz * in_plane + (long long)iy * a.wd + ix);
    sx[i] = v;
  }
}

// offset of tap k = (kz*3 + ky)*3 + kx inside the staged rows (relative to the row of this warp and the voxel column); taps >= 27
// are the zero padding of K: they read a valid address and are multiplied by a zero weight / masked
__device__ __forceinline__ int stem_tap_offset(int k, int Wa, int planar) {
  if (k >= (planar ? 9 : 27)) return 0;
  const int kz = k / 9, ky = (k / 3) % 3, kx = k % 3;
  return (kz * 10 + ky) * Wa + kx;
}

// ------------------------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------------------------
// PLANAR (k = (1,3,3)) is a template parameter: with a run-time tap count the K loop stays rolled and the B fragments / tap offsets
// it indexes end up in local memory (one LDL per MMA operand -- what made the first version latency bound, IPC 0.17 per scheduler).
template <bool PLANAR>
__global__ void __launch_bounds__(256, 3) stem_fwd_mma_kernel(const StemArgs a) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int Wp = (a.wd + 15) / 16 * 16;  // row length rounded up to whole 16-voxel M tiles
  const int Wa = Wp + 2;
  float* sx = reinterpret_cast<float*>(smem_raw);                                  // [3][10][Wa]
  uint8_t* sout = smem_raw + (((size_t)30 * Wa * sizeof(float) + 15) & ~size_t(15));  // [8 warps][16 rows][kStemRowPad]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  constexpr int ntaps = PLANAR ? 9 : 27;
  constexpr int ksteps = PLANAR ? 1 : 2;  // K = taps padded to 16 / 32

  // B fragments: B[k = tap][n = co] = W[co][tap], hi / lo split; b0 = (k = 2t, 2t+1), b1 = (k = 2t+8, 2t+9), n = g
  uint32_t bhi[2][4][2], blo[2][4][2];
#pragma unroll
  for (int ks = 0; ks < ksteps; ++ks)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k0 = ks * 16 + h * 8 + 2 * t, co = nt * 8 + g;
        const float w0 = k0 < ntaps ? __ldg(a.w + co * ntaps + k0) : 0.f;
        const float w1 = k0 + 1 < ntaps ? __ldg(a.w + co * ntaps + k0 + 1) : 0.f;
        split_bf16x2(w0, w1, bhi[ks][nt][h], blo[ks][nt][h]);
      }
  // this thread's 8 tap offsets: index (ks, h, j) -> k = ks*16 + h*8 + 2t + j
  int koff[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) koff[i] = stem_tap_offset((i >> 2) * 16 + ((i >> 1) & 1) * 8 + 2 * t + (i & 1), Wa, PLANAR);
  float bias[4][2];
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    bias[nt][0] = a.bias ? __ldg(a.bias + nt * 8 + 2 * t) : 0.f;
    bias[nt][1] = a.bias ? __ldg(a.bias + nt * 8 + 2 * t + 1) : 0.f;
  }

  const int ytiles = (a.h + 7) / 8;
  const long long tiles = (long long)a.n * a.d * ytiles;
  uint8_t* mine = sout + (size_t)warp * 16 * kStemRowPad;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int yt = (int)(tile % ytiles);
    const long long r = tile / ytiles;
    const int oz = (int)(r % a.d), nn = (int)(r / a.d);
    const int oy0 = yt * 8;
    __syncthreads();
    stem_stage_rows(a, sx, Wa, nn, oz, oy0);
    __syncthreads();
    const int oy = oy0 + warp;
    if (oy >= a.h) continue;
    const float* row = sx + warp * Wa;
    __nv_bfloat16* yrow = a.y + ((((long long)nn * a.d + oz) * a.h + oy) * a.wd) * a.ldy;
    for (int x0 = 0; x0 < a.wd; x0 += 16) {
      // A fragments: a0 = (row g, k 2t..), a1 = (row g+8, k 2t..), a2 = (row g, k 2t+8..), a3 = (row g+8, k 2t+8..)
      uint32_t ahi[2][4], alo[2][4];
#pragma unroll
      for (int ks = 0; ks < ksteps; ++ks)
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
          for (int rr = 0; rr < 2; ++rr) {
            const float* p = row + x0 + g + 8 * rr;
            const float v0 = p[koff[ks * 4 + h * 2]], v1 = p[koff[ks * 4 + h * 2 + 1]];
            split_bf16x2(v0, v1, ahi[ks][h * 2 + rr], alo[ks][h * 2 + rr]);
          }
      float acc[4][4];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        acc[nt][0] = acc[nt][2] = bias[nt][0];
        acc[nt][1] = acc[nt][3] = bias[nt][1];
      }
#pragma unroll
      for (int ks = 0; ks < ksteps; ++ks) {
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          mma_bf16_16816(acc[nt], ahi[ks], bhi[ks][nt][0], bhi[ks][nt][1]);
          mma_bf16_16816(acc[nt], alo[ks], bhi[ks][nt][0], bhi[ks][nt][1]);
          mma_bf16_16816(acc[nt], ahi[ks], blo[ks][nt][0], blo[ks][nt][1]);
        }
      }
      // activation, bf16, transpose through shared memory so that a thread writes 16 contiguous bytes (8 channels of a voxel)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float z = acc[nt][i];
          if (a.act == REHR_ACT_RELU) z = z > 0.f ? z : 0.f;
          if (a.act == REHR_ACT_LRELU) z = z > 0.f ? z : z * a.slope;
          acc[nt][i] = z;
        }
        *reinterpret_cast<uint32_t*>(mine + g * kStemRowPad + (nt * 8 + 2 * t) * 2) = pack16x2(acc[nt][0], acc[nt][1], a.y_f16);
        *reinterpret_cast<uint32_t*>(mine + (g + 8) * kStemRowPad + (nt * 8 + 2 * t) * 2) = pack16x2(acc[nt][2], acc[nt][3], a.y_f16);
      }
      if (a.range != nullptr) {  // the voxels x0 + g and x0 + g + 8 that are stored below
        uint32_t cnt = 0, mbits = 0;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          if (x0 + g < a.wd) { range_fold(acc[nt][0], cnt, mbits); range_fold(acc[nt][1], cnt, mbits); }
          if (x0 + g + 8 < a.wd) { range_fold(acc[nt][2], cnt, mbits); range_fold(acc[nt][3], cnt, mbits); }
        }
        range_flush(a.range, cnt, mbits);
      }
      __syncwarp();
#pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        const int vr = g + 8 * rr;
        const uint4 u = *reinterpret_cast<const uint4*>(mine + vr * kStemRowPad + t * 16);
        if (x0 + vr < a.wd) *reinterpret_cast<uint4*>(yrow + (long long)(x0 + vr) * a.ldy + t * 8) = u;
      }
      __syncwarp();
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// weight gradient
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], const void* smem_ptr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(smem_ptr)));
}

template <bool PLANAR>
__global__ void __launch_bounds__(256, 3) stem_wgrad_mma_kernel(const StemArgs a) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int Wp = (a.wd + 15) / 16 * 16;
  const int Wa = Wp + 2;
  float* sx = reinterpret_cast<float*>(smem_raw);                                  // [3][10][Wa]
  uint8_t* sdy = smem_raw + (((size_t)30 * Wa * sizeof(float) + 15) & ~size_t(15));   // [8 warps][2 buffers][16 rows][kStemRowPad]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  // A[m = tap][k = voxel]: a0 = (tap mt*16+g, v 2t..2t+1), a1 = (tap +8, same v), a2 = (tap, v 2t+8..), a3 = (tap +8, v 2t+8..)
  int toff[4];     // staged-row offsets of the taps g, g+8, g+16, g+24
  float tmask[4];  // 0 for the padding taps >= 27
  constexpr int ntaps = PLANAR ? 9 : 27;
  constexpr int mtiles = PLANAR ? 1 : 2;  // taps padded to 16 / 32
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    toff[i] = stem_tap_offset(g + 8 * i, Wa, PLANAR);
    tmask[i] = (g + 8 * i) < ntaps ? 1.f : 0.f;
  }
  float acc[2][4][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[mt][nt][i] = 0.f;

  const int ytiles = (a.h + 7) / 8;
  const long long tiles = (long long)a.n * a.d * ytiles;
  uint8_t* mybuf = sdy + (size_t)warp * 2 * 16 * kStemRowPad;
  // per-lane part of the dY staging: 16 voxels x 64 B = 64 x 16 B pieces, two per lane
  const int pv0 = lane >> 2, pc = lane & 3;  // piece (voxel pv0 / pv0 + 8, 16-byte column pc)
  // ldmatrix source row of this lane: matrix mi = lane / 8 -> (voxel half mi & 1, n-tile pair member mi >> 1), row lane % 8
  const int lm_v = (lane >> 3 & 1) * 8 + (lane & 7), lm_c = (lane >> 4) * 8;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int yt = (int)(tile % ytiles);
    const long long r = tile / ytiles;
    const int oz = (int)(r % a.d), nn = (int)(r / a.d);
    const int oy0 = yt * 8;
    __syncthreads();
    stem_stage_rows(a, sx, Wa, nn, oz, oy0);
    __syncthreads();
    const int oy = oy0 + warp;
    if (oy >= a.h) continue;
    const float* row = sx + warp * Wa;
    const __nv_bfloat16* dyrow = a.y + ((((long long)nn * a.d + oz) * a.h + oy) * a.wd) * a.ldy;
    const int steps = Wp / 16;
    // software pipeline: the dY pieces of step s + 1 are loaded into registers while step s computes
    uint4 nxt[2];
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      const int v = pv0 + 8 * rr;
      nxt[rr] = v < a.wd ? __ldcs(reinterpret_cast<const uint4*>(dyrow + (long long)v * a.ldy + pc * 8)) : make_uint4(0, 0, 0, 0);
    }
    for (int s = 0; s < steps; ++s) {
      const int x0 = s * 16;
      uint8_t* buf = mybuf + (size_t)(s & 1) * 16 * kStemRowPad;
#pragma unroll
      for (int rr = 0; rr < 2; ++rr) *reinterpret_cast<uint4*>(buf + (pv0 + 8 * rr) * kStemRowPad + pc * 16) = nxt[rr];
      if (s + 1 < steps) {
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
          const int v = x0 + 16 + pv0 + 8 * rr;
          nxt[rr] = v < a.wd ? __ldcs(reinterpret_cast<const uint4*>(dyrow + (long long)v * a.ldy + pc * 8)) : make_uint4(0, 0, 0, 0);
        }
      }
      __syncwarp();
      // B fragments (dY, exact bf16): n-tile pair p -> r0 = b0[2p], r1 = b1[2p], r2 = b0[2p+1], r3 = b1[2p+1]
      uint32_t bfr[2][4];
#pragma unroll
      for (int p = 0; p < 2; ++p) ldmatrix_x4_trans(bfr[p], buf + lm_v * kStemRowPad + (p * 16 + lm_c) * 2);
      // A fragments (im2col of the fp32 rows, hi / lo)
#pragma unroll
      for (int mt = 0; mt < mtiles; ++mt) {
        uint32_t ahi[4], alo[4];
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
          for (int rr = 0; rr < 2; ++rr) {
            const int ti = mt * 2 + rr;
            const float* p = row + toff[ti] + x0 + 2 * t + 8 * h;
            split_bf16x2(p[0] * tmask[ti], p[1] * tmask[ti], ahi[h * 2 + rr], alo[h * 2 + rr]);
          }
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const uint32_t b0 = bfr[nt >> 1][(nt & 1) * 2], b1 = bfr[nt >> 1][(nt & 1) * 2 + 1];
          mma_bf16_16816(acc[mt][nt], ahi, b0, b1);
          mma_bf16_16816(acc[mt][nt], alo, b0, b1);
        }
      }
    }
  }
  // cross-warp sum through shared memory: red[8][32 taps][33]
  __syncthreads();
  float* red = reinterpret_cast<float*>(smem_raw);
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const int tap = mt * 16 + g, co = nt * 8 + 2 * t;
      red[(warp * 32 + tap) * 33 + co] = acc[mt][nt][0];
      red[(warp * 32 + tap) * 33 + co + 1] = acc[mt][nt][1];
      red[(warp * 32 + tap + 8) * 33 + co] = acc[mt][nt][2];
      red[(warp * 32 + tap + 8) * 33 + co + 1] = acc[mt][nt][3];
    }
  __syncthreads();
  for (int i = threadIdx.x; i < ntaps * 32; i += 256) {
    const int tap = i / 32, co = i % 32;
    float sum = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) sum += red[(w * 32 + tap) * 33 + co];
    a.ws[((long long)blockIdx.x * 27 + tap) * 32 + co] = sum;
  }
}

// ws [blocks][27][32] -> dw [32][ntaps]; block = one tap: 32 channels x 8 slices of the partial list, fixed order
__global__ void __launch_bounds__(256) stem_wgrad_reduce_kernel(const float* ws, int blocks, float* dw, int accumulate, int ntaps) {
  __shared__ float red[8][33];
  const int co = threadIdx.x & 31, slice = threadIdx.x >> 5, tap = blockIdx.x;
  float s = 0.f;
  for (int b = slice; b < blocks; b += 8) s += ws[((long long)b * 27 + tap) * 32 + co];
  red[slice][co] = s;
  __syncthreads();
  if (slice == 0) {
    float tsum = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) tsum += red[k][co];
    float* d = dw + co * ntaps + tap;
    *d = accumulate ? *d + tsum : tsum;
  }
}

static size_t stem_smem_bytes(int wd, bool wgrad) {
  const int Wp = (wd + 15) / 16 * 16;
  const size_t rows = (((size_t)30 * (Wp + 2) * sizeof(float)) + 15) & ~size_t(15);
  const size_t tail = (size_t)8 * (wgrad ? 2 : 1) * 16 * kStemRowPad;
  const size_t red = wgrad ? (size_t)8 * 32 * 33 * sizeof(float) : 0;
  return std::max(rows + tail, red);
}

template <typename K>
static int stem_set_smem(K kernel, size_t smem, size_t* cached_per_device) {
  size_t* cached = cached_per_device + current_device();
  if (smem > 48 * 1024 && smem > *cached) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      g_last_cuda_error = (int)e;
      return REHR_CUDA_ERROR;
    }
    *cached = smem;
  }
  return REHR_OK;
}

static constexpr int kStemWgradBlocks = 444;  // 3 x 148 (launch bound: 3 blocks per SM)

bool stem_mma_supported(int cin, int cout, int wd) { return cin == 1 && cout == 32 && stem_smem_bytes(wd, true) <= 160 * 1024; }
size_t stem_mma_wgrad_workspace() { return (size_t)kStemWgradBlocks * 27 * 32 * sizeof(float); }

int launch_stem_fwd_mma(const float* x, const float* w, const float* bias, __nv_bfloat16* y, long long ldy, int y_f16, int n, int d, int h,
                        int wd, int act, float slope, int planar, cudaStream_t stream) {
  StemArgs a;
  a.planar = planar;
  a.y_f16 = y_f16;
  a.range = range_target(y_f16);
  a.x = x; a.w = w; a.bias = bias; a.y = y; a.ldy = ldy; a.ws = nullptr;
  a.n = n; a.d = d; a.h = h; a.wd = wd; a.act = act; a.slope = slope;
  const size_t smem = stem_smem_bytes(wd, false);
  static size_t cached[2 * kMaxDevices] = {};
  int rc = planar ? stem_set_smem(stem_fwd_mma_kernel<true>, smem, cached + kMaxDevices) : stem_set_smem(stem_fwd_mma_kernel<false>, smem, cached);
  if (rc != REHR_OK) return rc;
  const long long tiles = (long long)n * d * ((h + 7) / 8);
  const int blocks = (int)std::max<long long>(1, std::min<long long>(tiles, (long long)sm_count() * 3));
  if (planar) stem_fwd_mma_kernel<true><<<blocks, 256, smem, stream>>>(a);
  else stem_fwd_mma_kernel<false><<<blocks, 256, smem, stream>>>(a);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int launch_stem_wgrad_mma(const float* x, const __nv_bfloat16* dy, long long lddy, int n, int d, int h, int wd, float* dw, int accumulate,
                          float* ws, int planar, cudaStream_t stream) {
  StemArgs a;
  a.planar = planar;
  a.y_f16 = 0;
  a.range = nullptr;
  a.x = x; a.w = nullptr; a.bias = nullptr; a.y = const_cast<__nv_bfloat16*>(dy); a.ldy = lddy; a.ws = ws;
  a.n = n; a.d = d; a.h = h; a.wd = wd; a.act = 0; a.slope = 0.f;
  const size_t smem = stem_smem_bytes(wd, true);
  static size_t cached[2 * kMaxDevices] = {};
  int rc = planar ? stem_set_smem(stem_wgrad_mma_kernel<true>, smem, cached + kMaxDevices) : stem_set_smem(stem_wgrad_mma_kernel<false>, smem, cached);
  if (rc != REHR_OK) return rc;
  const long long tiles = (long long)n * d * ((h + 7) / 8);
  const int blocks = (int)std::max<long long>(1, std::min<long long>(tiles, (long long)kStemWgradBlocks));
  if (planar) stem_wgrad_mma_kernel<true><<<blocks, 256, smem, stream>>>(a);
  else stem_wgrad_mma_kernel<false><<<blocks, 256, smem, stream>>>(a);
  REHR_CHECK_LAUNCH();
  stem_wgrad_reduce_kernel<<<planar ? 9 : 27, 256, 0, stream>>>(ws, blocks, dw, accumulate, planar ? 9 : 27);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

}  // namespace rehr
