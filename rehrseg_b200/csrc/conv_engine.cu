// Dense convolution engine for sm_100a: "tapped GEMM" kernels on tcgen05 / TMEM with TMA-staged
// channels-last bf16 tiles.
//
//   fwd / dgrad :  out[o, n] = act( sum_taps sum_c  T_j(in)[o, c] * Wp[n][j][c] + bias[n] )
//                  (M = 128 output voxels per tile, N = output channels, K = taps x in-channels;
//                   A and B are K-major SW128/64/32 tiles written by TMA, accumulators in TMEM)
//   wgrad       :  D[(j, cm), cn] = sum_o  T_j(X)[o, cm] * Y[o, cn]
//                  (both operands MN-major views of the same [voxel][channel] TMA tiles, K = voxels)
//
// T_j(.) is "the input seen through tap j": a shifted (and, for strided convs, parity-decimated) window of
// the NDHWC tensor that one 5-D TMA box load produces directly, zero-filled outside the volume -- so there
// is no im2col buffer and padding costs nothing.  Strides are handled by one tensor map per input parity
// class (doubled pitches + base offset) instead of TMA element strides.
//
// Reference call sites replaced: every torch.nn.Conv3d / ConvTranspose3d / Conv2d on the hot path
// (SURVEY.md section 2.2; models/seg_model.py:174-199, models/FLAVR/FLAVR_arch.py:24-88,
// models/FLAVR/resnet_3D.py:19-33).
#include "engine.h"
#include "ptx.cuh"
#include "reduce.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

namespace rehr {

// ------------------------------------------------------------------------------------------------
// Host: driver entry point for tensor-map encoding (no link-time dependency on libcuda).
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static std::once_flag g_encode_once;
thread_local int g_last_cuda_error = 0;

static EncodeTiledFn get_encode() {
  std::call_once(g_encode_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    if (e == cudaSuccess && q == cudaDriverEntryPointSuccess) g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  });
  return g_encode;
}

int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return 0;
  return dev;
}

int sm_count() {
  static int n[kMaxDevices] = {};
  const int dev = current_device();
  if (n[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) return 148;
    n[dev] = v;
  }
  return n[dev];
}

// Dynamic shared memory a tensor-core conv CTA may plan with.  The persistent conv kernels run one CTA per SM and would otherwise
// take all 227 KB, which keeps every other kernel off the SM (each resident CTA needs its static shared memory + 1 KB): leaving
// a few KB free lets the HBM-bound InstanceNorm passes of the other sample stream become resident NEXT to a conv CTA
// (functional.py, sample streams).  REHR_SMEM_RESERVE_KB overrides the reserve (0 = the kernels take everything).
size_t smem_budget() {
  static size_t v = 0;
  if (v == 0) {
    const char* e = getenv("REHR_SMEM_RESERVE_KB");
    int kb = e ? atoi(e) : kDefaultSmemReserveKB;
    if (kb < 0) kb = 0;
    if (kb > 64) kb = 64;
    v = (size_t)(227 - kb) * 1024;
  }
  return v;
}

static CUtensorMapSwizzle swizzle_for_chunk(int chunk) {
  return chunk == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (chunk == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}

// 5-D map over a (possibly parity-decimated) NDHWC bf16 tensor.  dims/pitches in elements.
static int encode_act_map(CUtensorMap* m, const void* base, int C, const int ext[4], const long long pitch[4],
                          int chunk, const int box[4]) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return REHR_CUDA_ERROR;
  cuuint64_t gdim[5] = {(cuuint64_t)C, (cuuint64_t)ext[0], (cuuint64_t)ext[1], (cuuint64_t)ext[2], (cuuint64_t)ext[3]};
  cuuint64_t gstr[4] = {(cuuint64_t)pitch[0] * 2, (cuuint64_t)pitch[1] * 2, (cuuint64_t)pitch[2] * 2,
                        (cuuint64_t)pitch[3] * 2};
  cuuint32_t bdim[5] = {(cuuint32_t)chunk, (cuuint32_t)box[0], (cuuint32_t)box[1], (cuuint32_t)box[2], (cuuint32_t)box[3]};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return REHR_BAD_ALIGNMENT;
  for (int i = 0; i < 4; ++i)
    if ((gstr[i] & 15) != 0) return REHR_BAD_ALIGNMENT;
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(base), gdim, gstr, bdim, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for_chunk(chunk), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    g_last_cuda_error = (int)r;
    return REHR_CUDA_ERROR;
  }
  return REHR_OK;
}

// 2-D map over the packed weight matrix [rows][K] bf16 (K contiguous).
static int encode_weight_map(CUtensorMap* m, const void* base, long long K, int rows, int chunk, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return REHR_CUDA_ERROR;
  cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)K * 2};
  cuuint32_t bdim[2] = {(cuuint32_t)chunk, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (gstr[0] & 15) != 0) return REHR_BAD_ALIGNMENT;
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, bdim, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for_chunk(chunk), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    g_last_cuda_error = (int)r;
    return REHR_CUDA_ERROR;
  }
  return REHR_OK;
}

// Generic bf16 tiled tensor map (used by the marching kernel): dims / strides innermost first, strides in bytes.
int encode_tiled_bf16(CUtensorMap* m, const void* base, int rank, const unsigned long long* gdim,
                      const unsigned long long* gstride_bytes, const unsigned* box, int swizzle_bytes) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return REHR_CUDA_ERROR;
  cuuint64_t gd[5], gs[4];
  cuuint32_t bd[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gd[i] = gdim[i];
    bd[i] = box[i];
    es[i] = 1;
  }
  for (int i = 0; i + 1 < rank; ++i) {
    gs[i] = gstride_bytes[i];
    if ((gs[i] & 15) != 0) return REHR_BAD_ALIGNMENT;
  }
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return REHR_BAD_ALIGNMENT;
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : (swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bd, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    g_last_cuda_error = (int)r;
    return REHR_CUDA_ERROR;
  }
  return REHR_OK;
}

// ------------------------------------------------------------------------------------------------
// Host: tap tables.
// ------------------------------------------------------------------------------------------------
static inline int floordiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }
static inline int posmod(int a, int b) { return a - floordiv(a, b) * b; }

// Taps of the forward conv  out[o] += W[k] in[o*s + k - p]  (also used by wgrad for the X operand).
// Each distinct input parity class gets its own tensor map slot.
int build_fwd_taps(const rehr_conv_desc& cd, const rehr_tensor& in, TapPlan* plan) {
  plan->num_maps = 0;
  plan->num_taps = 0;
  plan->weight_taps = cd.kd * cd.kh * cd.kw;
  const int s[3] = {cd.sw, cd.sh, cd.sd}, p[3] = {cd.pw, cd.ph, cd.pd};
  const int isz[3] = {in.w, in.h, in.d};
  for (int kd = 0; kd < cd.kd; ++kd)
    for (int kh = 0; kh < cd.kh; ++kh)
      for (int kw = 0; kw < cd.kw; ++kw) {
        const int kk[3] = {kw, kh, kd};
        int r[3], q[3], ext[3];
        bool dead = false;
        for (int a = 0; a < 3; ++a) {
          const int e = kk[a] - p[a];
          r[a] = posmod(e, s[a]);
          q[a] = floordiv(e, s[a]);
          ext[a] = (isz[a] - r[a] + s[a] - 1) / s[a];
          if (ext[a] <= 0) dead = true;
        }
        if (dead) continue;  // every read of this tap is outside the volume
        int id = -1;
        for (int m = 0; m < plan->num_maps; ++m)
          if (plan->map_r[m][0] == r[0] && plan->map_r[m][1] == r[1] && plan->map_r[m][2] == r[2]) id = m;
        if (id < 0) {
          if (plan->num_maps >= kMaxMaps) return REHR_UNSUPPORTED;
          id = plan->num_maps++;
          for (int a = 0; a < 3; ++a) {
            plan->map_r[id][a] = r[a];
            plan->map_ext[id][a] = ext[a];
            plan->map_s[id][a] = s[a];
          }
        }
        if (plan->num_taps >= kMaxTaps) return REHR_UNSUPPORTED;
        Tap& t = plan->taps[plan->num_taps++];
        t.map_id = id;
        t.dw = q[0];
        t.dh = q[1];
        t.dd = q[2];
        t.widx = (kd * cd.kh + kh) * cd.kw + kw;
      }
  return REHR_OK;
}

// Taps of one output parity class (rw, rh, rd) of the input-gradient / transposed conv:
//   dx[i] += W[k] dy[(i + p - k) / s]   for the k with (i + p - k) % s == 0.
// The source (dy) is always read un-decimated, so a single map is used.
int build_dgrad_taps(const rehr_conv_desc& cd, const int cls[3], TapPlan* plan) {
  plan->num_maps = 1;
  for (int a = 0; a < 3; ++a) {
    plan->map_r[0][a] = 0;
    plan->map_s[0][a] = 1;
    plan->map_ext[0][a] = 0;  // filled by the caller from dy dims
  }
  plan->num_taps = 0;
  plan->weight_taps = cd.kd * cd.kh * cd.kw;
  const int s[3] = {cd.sw, cd.sh, cd.sd}, p[3] = {cd.pw, cd.ph, cd.pd};
  for (int kd = 0; kd < cd.kd; ++kd)
    for (int kh = 0; kh < cd.kh; ++kh)
      for (int kw = 0; kw < cd.kw; ++kw) {
        const int kk[3] = {kw, kh, kd};
        int q[3];
        bool ok = true;
        for (int a = 0; a < 3; ++a) {
          const int e = cls[a] + p[a] - kk[a];
          if (posmod(e, s[a]) != 0) ok = false;
          q[a] = floordiv(e, s[a]);
        }
        if (!ok) continue;
        if (plan->num_taps >= kMaxTaps) return REHR_UNSUPPORTED;
        Tap& t = plan->taps[plan->num_taps++];
        t.map_id = 0;
        t.dw = q[0];
        t.dh = q[1];
        t.dd = q[2];
        t.widx = (kd * cd.kh + kh) * cd.kw + kw;
      }
  return REHR_OK;
}

static int pow2ceil(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// Pick a (bw, bh, bd, bn) box with bw*bh*bd*bn == vox (a power of two): grow the dims round-robin so the
// box stays compact (best halo reuse in L2), never beyond the next power of two of each extent.
void choose_box(int W, int H, int D, int N, int vox, int box[4]) {
  const int lim[4] = {pow2ceil(W), pow2ceil(H), pow2ceil(D), pow2ceil(N)};
  box[0] = box[1] = box[2] = box[3] = 1;
  int prod = 1;
  while (prod < vox) {
    bool grew = false;
    for (int a = 0; a < 3 && prod < vox; ++a)
      if (box[a] * 2 <= lim[a]) {
        box[a] *= 2;
        prod *= 2;
        grew = true;
      }
    if (!grew) {  // spatial extent exhausted: span samples (rows past the batch are zero-filled and masked)
      box[3] *= 2;
      prod *= 2;
    }
  }
  (void)lim;
}

static int chunk_for_channels(int c) {
  if (c % 64 == 0) return 64;
  if (c % 32 == 0) return 32;
  if (c % 16 == 0) return 16;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Device: forward / dgrad kernel
// ------------------------------------------------------------------------------------------------
// warp0 TMA, warp1 MMA (+TMEM alloc), warps 2..9 epilogue: two warps per TMEM lane quarter (warp % 4), taking alternate 16-column
// chunks.  With one epilogue warp per scheduler every instruction latency of the drain was exposed (ncu: IPC 0.15, 2.2k clk per
// chunk) and small-K tiles (transposed convs, stride-2 stage entries) were bound by it.
static constexpr int kFwdThreads = 320;
static constexpr int kFwdEpiThreads = 256;
static constexpr int kWgradThreads = 192;  // conv_wgrad_kernel: warp0 TMA, warp1 MMA, warps 2..5 drain
static constexpr int kMaxStages = 8;

struct alignas(64) FwdParams {
  CUtensorMap a_map[kMaxMaps];
  CUtensorMap b_map;
  int2 taps[kMaxTaps];  // x = map_id | (dw+128)<<8 | (dh+128)<<16 | (dd+128)<<24 ; y = widx
  int num_taps;
  int box[4];      // bw bh bd bn (product 128)
  int tiles[4];    // boxes per dim
  int n_tiles;     // Cout tiles
  int BN;          // output channels per tile (multiple of 16, <= 256)
  int BK;          // in-channel chunk 64/32/16
  int cin_chunks;
  int cin;
  int stages;
  int tmem_cols;
  // output
  void* out;
  int out_f32;
  int out_f16;     // 16-bit output format (rehr_dtype of the output tensor) when !out_f32
  int in_f16;      // operand format of the input tensor AND of the packed weights
  // scatter epilogue only: optional second copy of the result in another buffer / 16-bit format (the bf16 twin of an fp16
  // up-sampled tensor inside the [up | skip] buffer that the consumer's weight gradient reads), written from the same registers
  void* out2;
  long long out2_ld;
  int out2_f16;
  RangeSlot* range;  // fp16 saturation record of the stored values (rehr_range_sink), null = not checked
  long long out_ld;
  int O[4];        // class-local output extents (w h d n)
  int os[3], oo[3];  // actual coord = o*os + oo (w h d)
  int AO[3];       // actual output tensor extents (w h d)
  int cout;
  const float* bias;
  int act;
  float slope;
  float* stats;    // [m_tile][cout][2] or null
  // "scatter" epilogue of a kernel == stride transposed conv computed as ONE GEMM with N = classes x cout:
  // column block (cls, co) of row (input voxel i) is output voxel i*s + r(cls), channel co.  0 = off.
  int sc_cout;
  int sc_s[3];     // stride per dim (w h d)
  long long sc_off[8];  // output voxel offset of class cls = (rd * AO[1] + rh) * AO[0] + rw (at most 8 classes)
  // split-K for layers with fewer output tiles than SMs (the <= 8^3 bottleneck stages stream 2-5 MB of weights and taps
  // through ONE or TWO SMs otherwise): work item = (tile, split); a split accumulates its share of the (tap, Cin-chunk)
  // K blocks and stores raw fp32 partials [split][tile][128][BN]; conv_splitk_finish_kernel sums them and runs the epilogue.
  int ksplit;
  float* partial;
  int* err;
};

__device__ __forceinline__ float apply_act(float v, int act, float slope) {
  if (act == REHR_ACT_RELU) return v > 0.f ? v : 0.f;
  if (act == REHR_ACT_LRELU) return v > 0.f ? v : v * slope;
  return v;
}

// bias + InstanceNorm partial sums + activation + store of one 16-column chunk of one accumulator row (non-scatter epilogue)
template <bool RC>
__device__ __forceinline__ void finish_chunk(const FwdParams& p, float (&f)[16], bool valid, long long vox, int nbase, int c0,
                                             int lane, float* mypart);

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}

// One K block = KSTEPS tcgen05.mma with compile-time descriptor increments.  Issued from warp-uniform control flow by an
// elected lane so that the descriptors stay in uniform registers: with `if (lane == 0)` and run-time descriptor arithmetic a
// single thread needs 120-280 clk per MMA (tools/umma_rate2.cu), which bounds every N <= 256 tile of this kernel.
template <int KSTEPS>
__device__ __forceinline__ void issue_kblock(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t a_hi, uint32_t b_hi,
                                             uint32_t idesc, bool first, uint32_t a_step, uint32_t b_step) {
#pragma unroll
  for (int k = 0; k < KSTEPS; ++k) {
    const uint64_t ad = ((uint64_t)a_hi << 32) | (uint64_t)(a_lo + (uint32_t)k * a_step);
    const uint64_t bd = ((uint64_t)b_hi << 32) | (uint64_t)(b_lo + (uint32_t)k * b_step);
    umma_bf16(d_tmem, ad, bd, idesc, (first && k == 0) ? 0u : 1u);
  }
}

// RC: the fp16 saturation check of the stored values (p.range != null) is compiled in (see conv_tapped_gemm_kernel)
template <bool RC>
__device__ __forceinline__ void finish_chunk(const FwdParams& p, float (&f)[16], bool valid, long long vox, int nbase, int c0,
                                             int lane, float* mypart) {
  if (p.bias != nullptr) {
    if (nbase + c0 + 16 <= p.cout && ((nbase + c0) & 3) == 0) {
#pragma unroll
      for (int i = 0; i < 16; i += 4) {
        const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + nbase + c0 + i));
        f[i] += b4.x; f[i + 1] += b4.y; f[i + 2] += b4.z; f[i + 3] += b4.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int c = nbase + c0 + i;
        if (c < p.cout) f[i] += __ldg(p.bias + c);
      }
    }
  }
  if (p.stats != nullptr) {
    float s1[16], s2[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const float x = valid ? f[i] : 0.f;
      s1[i] = x;
      s2[i] = x * x;
    }
    warp_colsum16(s1, lane);
    warp_colsum16(s2, lane);
    if ((lane & 1) == 0) {
      const int col = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
      mypart[c0 + col] = s1[0];
      mypart[256 + c0 + col] = s2[0];
    }
  }
  if (valid) {
#pragma unroll
    for (int i = 0; i < 16; ++i) f[i] = apply_act(f[i], p.act, p.slope);
    const int cbase = nbase + c0;
    if (p.out_f32) {
      float* o = reinterpret_cast<float*>(p.out) + vox * p.out_ld + cbase;
      if (cbase + 16 <= p.cout && (p.out_ld & 3) == 0) {
#pragma unroll
        for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(o + i) = make_float4(f[i], f[i + 1], f[i + 2], f[i + 3]);
      } else {
        for (int i = 0; i < 16; ++i)
          if (cbase + i < p.cout) o[i] = f[i];
      }
    } else {
      unsigned short* o = reinterpret_cast<unsigned short*>(p.out) + vox * p.out_ld + cbase;
      if constexpr (RC) range_check<16>(p.range, f, p.cout - cbase);
      if (cbase + 16 <= p.cout && (p.out_ld & 7) == 0) {
        uint4 lo, hi;
        lo.x = pack16x2(f[0], f[1], p.out_f16);
        lo.y = pack16x2(f[2], f[3], p.out_f16);
        lo.z = pack16x2(f[4], f[5], p.out_f16);
        lo.w = pack16x2(f[6], f[7], p.out_f16);
        hi.x = pack16x2(f[8], f[9], p.out_f16);
        hi.y = pack16x2(f[10], f[11], p.out_f16);
        hi.z = pack16x2(f[12], f[13], p.out_f16);
        hi.w = pack16x2(f[14], f[15], p.out_f16);
        reinterpret_cast<uint4*>(o)[0] = lo;
        reinterpret_cast<uint4*>(o)[1] = hi;
      } else {
        for (int i = 0; i < 16; ++i)
          if (cbase + i < p.cout) o[i] = pack16(f[i], p.out_f16);
      }
    }
  }
}

// RC: the fp16 saturation check of the stored values is compiled in; the default instantiation has no trace of it.
template <bool RC>
__global__ void __launch_bounds__(kFwdThreads, 1) conv_tapped_gemm_kernel(const __grid_constant__ FwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-B alignment of the dynamic window is required by the 128B swizzle atoms.
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t a_bytes = 128u * p.BK * 2u;
  const uint32_t b_bytes = (uint32_t)p.BN * p.BK * 2u;
  const uint32_t stage_bytes = a_bytes + b_bytes;
  uint8_t* tail = smem + (size_t)p.stages * stage_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_bar = full_bar + kMaxStages;
  uint64_t* tfull_bar = empty_bar + kMaxStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  float* part = reinterpret_cast<float*>(tmem_slot + 4);  // [2 acc][4 warps][2][256]

  if (warp == 0 && lane == 0) {
    for (int m = 0; m < kMaxMaps; ++m) tma_prefetch_desc(&p.a_map[m]);
    tma_prefetch_desc(&p.b_map);
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], kFwdEpiThreads / 32);
    }
    fence_mbar_init();
  } else if (warp == 1) {
    tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int m_tiles = p.tiles[0] * p.tiles[1] * p.tiles[2] * p.tiles[3];
  const int total_tiles = m_tiles * p.n_tiles;
  const int total_work = total_tiles * p.ksplit;
  const int kblocks = p.num_taps * p.cin_chunks;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int work = blockIdx.x; work < total_work; work += gridDim.x) {
        const int tile = work / p.ksplit, split = work - tile * p.ksplit;
        const int kb0 = (int)(((long long)kblocks * split) / p.ksplit), kb1 = (int)(((long long)kblocks * (split + 1)) / p.ksplit);
        const int n_tile = tile % p.n_tiles;
        int mt = tile / p.n_tiles;
        const int tw = mt % p.tiles[0];
        mt /= p.tiles[0];
        const int th = mt % p.tiles[1];
        mt /= p.tiles[1];
        const int td = mt % p.tiles[2];
        const int tn = mt / p.tiles[2];
        const int w0 = tw * p.box[0], h0 = th * p.box[1], d0 = td * p.box[2], n0 = tn * p.box[3];
        for (int kb = kb0; kb < kb1; ++kb) {
          const int j = kb / p.cin_chunks, cc = kb - j * p.cin_chunks;
          const int2 t = p.taps[j];
          const int map_id = t.x & 0xff;
          const int dw = ((t.x >> 8) & 0xff) - 128, dh = ((t.x >> 16) & 0xff) - 128, dd = ((t.x >> 24) & 0xff) - 128;
          const int kbase = t.y * p.cin;
          mbar_wait(&empty_bar[stage], phase ^ 1u, p.err, 1);
          uint8_t* sa = smem + (size_t)stage * stage_bytes;
          mbar_arrive_expect_tx(&full_bar[stage], stage_bytes);
          tma_load_5d(&p.a_map[map_id], &full_bar[stage], sa, cc * p.BK, w0 + dw, h0 + dh, d0 + dd, n0);
          tma_load_2d(&p.b_map, &full_bar[stage], sa + a_bytes, kbase + cc * p.BK, n_tile * p.BN);
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t idesc = make_idesc_16(128, p.BN, 0, 0, p.in_f16);
    const uint32_t row_bytes = (uint32_t)p.BK * 2u;
    const uint32_t layout = swizzle_layout_for_bytes((int)row_bytes);
    const uint32_t sbo = 8u * row_bytes;
    const uint32_t desc_hi = ((sbo >> 4) & 0x3FFFu) | (1u << 14) | (layout << 29);  // SBO, version 1, swizzle mode
    const uint32_t smem_lo = smem_u32(smem) >> 4, stage_lo = stage_bytes >> 4, a_lo_bytes = a_bytes >> 4;
    int stage = 0;
    uint32_t phase = 0;
    int iter = 0;
    for (int work = blockIdx.x; work < total_work; work += gridDim.x, ++iter) {
      const int split = work % p.ksplit;
      const int kb0 = (int)(((long long)kblocks * split) / p.ksplit), kb1 = (int)(((long long)kblocks * (split + 1)) / p.ksplit);
      const int acc = iter & 1;
      const uint32_t acc_phase = (uint32_t)(iter >> 1) & 1u;
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1u, p.err, 2);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.BN);
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&full_bar[stage], phase, p.err, 3);
        tc_fence_after();
        const uint32_t sa_lo = smem_lo + (uint32_t)stage * stage_lo;
        const uint32_t sb_lo = sa_lo + a_lo_bytes;
        if (elect_one()) {
          if (p.BK == 64) issue_kblock<4>(d_tmem, sa_lo, sb_lo, desc_hi, desc_hi, idesc, kb == kb0, 2u, 2u);
          else if (p.BK == 32) issue_kblock<2>(d_tmem, sa_lo, sb_lo, desc_hi, desc_hi, idesc, kb == kb0, 2u, 2u);
          else issue_kblock<1>(d_tmem, sa_lo, sb_lo, desc_hi, desc_hi, idesc, kb == kb0, 2u, 2u);
          umma_commit(&empty_bar[stage]);
          if (kb == kb1 - 1) umma_commit(&tfull_bar[acc]);
        }
        __syncwarp();
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else {
    // ===================== epilogue (warps 2..9) =====================
    const int q = warp & 3;          // TMEM lane quarter this warp may touch
    const int half = (warp - 2) >> 2;  // the two warps of a quarter take alternate 16-column chunks
    const int row = q * 32 + lane;   // accumulator row = voxel within the box
    const int et = threadIdx.x - 64; // 0..255
    int iter = 0;
    for (int work = blockIdx.x; work < total_work; work += gridDim.x, ++iter) {
      const int tile = work / p.ksplit, split = work - tile * p.ksplit;
      const int acc = iter & 1;
      const uint32_t acc_phase = (uint32_t)(iter >> 1) & 1u;
      const int n_tile = tile % p.n_tiles;
      const int m_tile = tile / p.n_tiles;
      int mt = m_tile;
      const int tw = mt % p.tiles[0];
      mt /= p.tiles[0];
      const int th = mt % p.tiles[1];
      mt /= p.tiles[1];
      const int td = mt % p.tiles[2];
      const int tn = mt / p.tiles[2];
      int r = row;
      const int ow = tw * p.box[0] + r % p.box[0];
      r /= p.box[0];
      const int oh = th * p.box[1] + r % p.box[1];
      r /= p.box[1];
      const int od = td * p.box[2] + r % p.box[2];
      r /= p.box[2];
      const int on = tn * p.box[3] + r;
      const bool valid = ow < p.O[0] && oh < p.O[1] && od < p.O[2] && on < p.O[3];
      const long long vox = (((long long)on * p.AO[2] + (od * p.os[2] + p.oo[2])) * p.AO[1] + (oh * p.os[1] + p.oo[1])) *
                                p.AO[0] + (ow * p.os[0] + p.oo[0]);
      const int nbase = n_tile * p.BN;
      float* mypart = part + ((acc * 4 + q) * 2) * 256;

      mbar_wait(&tfull_bar[acc], acc_phase, p.err, 4);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * p.BN);
      // scatter epilogue bookkeeping without per-chunk divisions: class / channel of this warp's first chunk, then +32 columns
      int sc_cls = 0, sc_co0 = 0;
      long long sc_ov0 = 0;
      if (p.sc_cout > 0) {
        const int col0 = nbase + half * 16;
        sc_cls = col0 / p.sc_cout;
        sc_co0 = col0 - sc_cls * p.sc_cout;
        sc_ov0 = (((long long)on * p.AO[2] + od * p.sc_s[2]) * p.AO[1] + oh * p.sc_s[1]) * p.AO[0] + ow * p.sc_s[0];
      }
      const int sc_ncls = p.sc_s[0] * p.sc_s[1] * p.sc_s[2];
      for (int c0 = half * 16; c0 < p.BN; c0 += 32) {
        uint32_t v[16];
        tmem_ld16(taddr + (uint32_t)c0, v);
        tmem_ld_wait();
        float f[16];
        if (p.sc_cout > 0) {
          // scatter epilogue: this 16-column chunk belongs to one output parity class
          const int cls = sc_cls, co0 = sc_co0;
          sc_co0 += 32;
          while (sc_co0 >= p.sc_cout) {
            sc_co0 -= p.sc_cout;
            ++sc_cls;
          }
          if (valid && cls < sc_ncls) {
            const long long ov = sc_ov0 + p.sc_off[cls];
#pragma unroll
            for (int i = 0; i < 16; ++i) f[i] = __uint_as_float(v[i]);
            if (p.bias != nullptr) {
#pragma unroll
              for (int i = 0; i < 16; i += 4) {
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + co0 + i));
                f[i] += b4.x; f[i + 1] += b4.y; f[i + 2] += b4.z; f[i + 3] += b4.w;
              }
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) f[i] = apply_act(f[i], p.act, p.slope);
            if constexpr (RC) range_check<16>(p.range, f);
            unsigned short* o = reinterpret_cast<unsigned short*>(p.out) + ov * p.out_ld + co0;
            uint4 lo, hi;
            lo.x = pack16x2(f[0], f[1], p.out_f16);
            lo.y = pack16x2(f[2], f[3], p.out_f16);
            lo.z = pack16x2(f[4], f[5], p.out_f16);
            lo.w = pack16x2(f[6], f[7], p.out_f16);
            hi.x = pack16x2(f[8], f[9], p.out_f16);
            hi.y = pack16x2(f[10], f[11], p.out_f16);
            hi.z = pack16x2(f[12], f[13], p.out_f16);
            hi.w = pack16x2(f[14], f[15], p.out_f16);
            reinterpret_cast<uint4*>(o)[0] = lo;
            reinterpret_cast<uint4*>(o)[1] = hi;
            if (p.out2 != nullptr) {
              unsigned short* o2 = reinterpret_cast<unsigned short*>(p.out2) + ov * p.out2_ld + co0;
              lo.x = pack16x2(f[0], f[1], p.out2_f16);
              lo.y = pack16x2(f[2], f[3], p.out2_f16);
              lo.z = pack16x2(f[4], f[5], p.out2_f16);
              lo.w = pack16x2(f[6], f[7], p.out2_f16);
              hi.x = pack16x2(f[8], f[9], p.out2_f16);
              hi.y = pack16x2(f[10], f[11], p.out2_f16);
              hi.z = pack16x2(f[12], f[13], p.out2_f16);
              hi.w = pack16x2(f[14], f[15], p.out2_f16);
              reinterpret_cast<uint4*>(o2)[0] = lo;
              reinterpret_cast<uint4*>(o2)[1] = hi;
            }
          }
          continue;
        }
        if (p.partial != nullptr) {  // split-K: raw fp32 partial, finished by conv_splitk_finish_kernel
          float4* o = reinterpret_cast<float4*>(p.partial + (((size_t)split * total_tiles + tile) * 128 + row) * p.BN + c0);
#pragma unroll
          for (int i = 0; i < 4; ++i)
            o[i] = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]), __uint_as_float(v[4 * i + 2]),
                               __uint_as_float(v[4 * i + 3]));
          continue;
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) f[i] = __uint_as_float(v[i]);
        finish_chunk<RC>(p, f, valid, vox, nbase, c0, lane, mypart);
      }
      // accumulator drained: hand the TMEM stage back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if (p.stats != nullptr && p.partial == nullptr) {
        named_bar_sync(1, kFwdEpiThreads);
        for (int c = et; c < p.BN; c += kFwdEpiThreads) {
          if (nbase + c < p.cout) {
            float a = 0.f, b = 0.f;
#pragma unroll
            for (int w = 0; w < 4; ++w) {
              a += part[((acc * 4 + w) * 2) * 256 + c];
              b += part[((acc * 4 + w) * 2 + 1) * 256 + c];
            }
            float* dst = p.stats + ((long long)m_tile * p.cout + nbase + c) * 2;
            dst[0] = a;
            dst[1] = b;
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// Second stage of split-K: one CTA of 128 threads per (output tile, 16-column chunk); thread = accumulator row; sums the `ksplit`
// raw partials and runs the same per-chunk epilogue (bias, InstanceNorm partial sums, activation, store) as the fused path.
template <bool RC>
__global__ void __launch_bounds__(128) conv_splitk_finish_kernel(const __grid_constant__ FwdParams p) {
  __shared__ float part[4 * 2 * 256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = threadIdx.x;
  const int tile = blockIdx.x;
  const int c0 = blockIdx.y * 16;
  const int total_tiles = gridDim.x;
  const int n_tile = tile % p.n_tiles;
  const int m_tile = tile / p.n_tiles;
  int mt = m_tile;
  const int tw = mt % p.tiles[0];
  mt /= p.tiles[0];
  const int th = mt % p.tiles[1];
  mt /= p.tiles[1];
  const int td = mt % p.tiles[2];
  const int tn = mt / p.tiles[2];
  int r = row;
  const int ow = tw * p.box[0] + r % p.box[0];
  r /= p.box[0];
  const int oh = th * p.box[1] + r % p.box[1];
  r /= p.box[1];
  const int od = td * p.box[2] + r % p.box[2];
  r /= p.box[2];
  const int on = tn * p.box[3] + r;
  const bool valid = ow < p.O[0] && oh < p.O[1] && od < p.O[2] && on < p.O[3];
  const long long vox = (((long long)on * p.AO[2] + (od * p.os[2] + p.oo[2])) * p.AO[1] + (oh * p.os[1] + p.oo[1])) * p.AO[0] +
                        (ow * p.os[0] + p.oo[0]);
  const int nbase = n_tile * p.BN;
  float* mypart = part + (warp * 2) * 256;
  float f[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) f[i] = 0.f;
  const float* src0 = p.partial + ((size_t)tile * 128 + row) * p.BN + c0;
  const size_t sstride = (size_t)total_tiles * 128 * p.BN;
#pragma unroll 4
  for (int s = 0; s < p.ksplit; ++s) {
    const float4* src = reinterpret_cast<const float4*>(src0 + (size_t)s * sstride);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 v = src[i];
      f[4 * i] += v.x; f[4 * i + 1] += v.y; f[4 * i + 2] += v.z; f[4 * i + 3] += v.w;
    }
  }
  finish_chunk<RC>(p, f, valid, vox, nbase, c0, lane, mypart);
  if (p.stats != nullptr) {
    __syncthreads();
    if (threadIdx.x < 16 && nbase + c0 + threadIdx.x < p.cout) {
      const int c = c0 + threadIdx.x;
      float a = 0.f, b = 0.f;
#pragma unroll
      for (int w = 0; w < 4; ++w) {
        a += part[(w * 2) * 256 + c];
        b += part[(w * 2 + 1) * 256 + c];
      }
      float* dst = p.stats + ((long long)m_tile * p.cout + nbase + c) * 2;
      dst[0] = a;
      dst[1] = b;
    }
  }
}

static size_t fwd_smem_tail_bytes() { return (2 * kMaxStages + 4) * 8 + 16 + 2 * 4 * 2 * 256 * 4; }

// Launch one tapped GEMM:  out(class) = act(sum_taps T_j(in) Wp + bias).
// `in_ext` are the input tensor extents (w h d n); O = class-local output extents; out coordinate
// transform (os, oo); AO = actual output extents.
int launch_tapped_gemm(const TapPlan& plan, const rehr_tensor& in, const void* w_packed, int w_rows,
                       const float* bias, const rehr_tensor& out, int out_f32, const int O[4], const int os[3],
                       const int oo[3], int act, float slope, float* stats, cudaStream_t stream, const int* scatter_s, void* ws,
                       size_t ws_bytes, size_t* ws_need, const rehr_tensor* out2) {
  const int cin = in.c;
  const int ncls = scatter_s ? scatter_s[0] * scatter_s[1] * scatter_s[2] : 1;
  const int cout = out.c * ncls;  // GEMM N: all parity classes side by side in scatter mode
  if (scatter_s && (out.c % 16 != 0 || out_f32 || stats != nullptr || out.ld % 8 != 0)) return REHR_UNSUPPORTED;
  const int BK = chunk_for_channels(cin);
  if (BK == 0) return REHR_UNSUPPORTED;
  if (in.ld % 8 != 0) return REHR_BAD_ALIGNMENT;
  if (plan.num_taps == 0) return REHR_UNSUPPORTED;
  (void)w_rows;

  FwdParams p;
  memset(&p, 0, sizeof(p));
  // N tiling: as few, as equal tiles as possible, each a multiple of 16 and <= 256.
  const int cout16 = (cout + 15) / 16 * 16;
  int n_tiles = (cout16 + 255) / 256;
  int BN = ((cout16 / 16 + n_tiles - 1) / n_tiles) * 16;
  p.n_tiles = n_tiles;
  p.BN = BN;
  p.BK = BK;
  p.cin = cin;
  p.cin_chunks = cin / BK;
  p.num_taps = plan.num_taps;
  choose_box(O[0], O[1], O[2], O[3], 128, p.box);
  for (int a = 0; a < 4; ++a) {
    p.tiles[a] = (O[a] + p.box[a] - 1) / p.box[a];
    p.O[a] = O[a];
  }
  if (stats != nullptr && p.box[3] != 1) return REHR_UNSUPPORTED;
  for (int a = 0; a < 3; ++a) {
    p.os[a] = os[a];
    p.oo[a] = oo[a];
  }
  p.AO[0] = out.w;
  p.AO[1] = out.h;
  p.AO[2] = out.d;
  p.out = out.ptr;
  p.out_f32 = out_f32;
  p.out_f16 = out.dtype == REHR_F16;
  p.in_f16 = in.dtype == REHR_F16;
  if (out2 != nullptr) {
    if (!scatter_s || out2->c != out.c || out2->ld % 8 != 0 || (reinterpret_cast<uintptr_t>(out2->ptr) & 15) != 0) return REHR_UNSUPPORTED;
    p.out2 = out2->ptr;
    p.out2_ld = out2->ld;
    p.out2_f16 = out2->dtype == REHR_F16;
  }
  p.range = range_target(!out_f32 && (p.out_f16 || (out2 != nullptr && p.out2_f16)));
  p.out_ld = out.ld;
  p.cout = cout;
  p.bias = bias;
  p.act = act;
  p.slope = slope;
  p.stats = stats;
  p.err = nullptr;
  if (scatter_s) {
    if (ncls > 8) return REHR_UNSUPPORTED;
    p.sc_cout = out.c;
    for (int a = 0; a < 3; ++a) p.sc_s[a] = scatter_s[a];
    for (int cls = 0; cls < ncls; ++cls) {
      const int rw = cls % scatter_s[0], rh = (cls / scatter_s[0]) % scatter_s[1], rd = cls / (scatter_s[0] * scatter_s[1]);
      p.sc_off[cls] = ((long long)rd * out.h + rh) * out.w + rw;
    }
  }
  int tc = 32;
  while (tc < 2 * BN) tc <<= 1;
  p.tmem_cols = tc;

  for (int j = 0; j < plan.num_taps; ++j) {
    const Tap& t = plan.taps[j];
    if (t.dw < -128 || t.dw > 127 || t.dh < -128 || t.dh > 127 || t.dd < -128 || t.dd > 127) return REHR_UNSUPPORTED;
    p.taps[j].x = (t.map_id & 0xff) | ((t.dw + 128) << 8) | ((t.dh + 128) << 16) | ((t.dd + 128) << 24);
    p.taps[j].y = t.widx;
  }
  // activation maps (one per parity class)
  const long long pitch_w = in.ld, pitch_h = (long long)in.w * in.ld, pitch_d = (long long)in.h * pitch_h,
                  pitch_n = (long long)in.d * pitch_d;
  const long long base_pitch[3] = {pitch_w, pitch_h, pitch_d};
  const int isz[3] = {in.w, in.h, in.d};
  for (int m = 0; m < kMaxMaps; ++m) {
    const int mm = m < plan.num_maps ? m : 0;
    int ext[4];
    long long pitch[4];
    long long off = 0;
    for (int a = 0; a < 3; ++a) {
      const int s = plan.map_s[mm][a], r = plan.map_r[mm][a];
      ext[a] = (isz[a] - r + s - 1) / s;
      pitch[a] = base_pitch[a] * s;
      off += (long long)r * base_pitch[a];
    }
    ext[3] = in.n;
    pitch[3] = pitch_n;
    const __nv_bfloat16* base = reinterpret_cast<const __nv_bfloat16*>(in.ptr) + off;
    int rc = encode_act_map(&p.a_map[m], base, cin, ext, pitch, BK, p.box);
    if (rc != REHR_OK) return rc;
  }
  {
    const long long K = (long long)plan.weight_taps * cin;
    int rc = encode_weight_map(&p.b_map, w_packed, K, cout, BK, BN);
    if (rc != REHR_OK) return rc;
  }
  const size_t stage_bytes = (size_t)128 * BK * 2 + (size_t)BN * BK * 2;
  const size_t budget = smem_budget() - 1024 - fwd_smem_tail_bytes();
  int stages = (int)std::min<size_t>(kMaxStages, budget / stage_bytes);
  if (stages < 2) return REHR_UNSUPPORTED;
  p.stages = stages;
  const size_t smem = 1024 + stages * stage_bytes + fwd_smem_tail_bytes();

  const bool rc = p.range != nullptr;
  if (rc)
    REHR_SET_MAX_SMEM_ONCE(conv_tapped_gemm_kernel<true>, 227 * 1024);
  else
    REHR_SET_MAX_SMEM_ONCE(conv_tapped_gemm_kernel<false>, 227 * 1024);
  const int total_tiles = p.tiles[0] * p.tiles[1] * p.tiles[2] * p.tiles[3] * p.n_tiles;
  // split-K when the output tiles cannot fill the machine and there is a long K loop to share
  const int kblocks = p.num_taps * p.cin_chunks;
  int ksplit = 1;
  if (!scatter_s && total_tiles * 4 <= sm_count() && kblocks >= 16) {
    ksplit = std::min(std::min(kblocks / 8, sm_count() / total_tiles), 32);
    if (ksplit < 2) ksplit = 1;
  }
  const size_t need = ksplit > 1 ? (size_t)ksplit * total_tiles * 128 * BN * sizeof(float) : 0;
  if (ws_need) {  // planning query only
    *ws_need = need;
    return REHR_OK;
  }
  if (ksplit > 1 && (ws == nullptr || ws_bytes < need)) ksplit = 1;  // no scratch supplied: single pass
  p.ksplit = ksplit;
  p.partial = ksplit > 1 ? reinterpret_cast<float*>(ws) : nullptr;
  const int grid = std::min(total_tiles * ksplit, sm_count());
  if (rc)
    conv_tapped_gemm_kernel<true><<<grid, kFwdThreads, smem, stream>>>(p);
  else
    conv_tapped_gemm_kernel<false><<<grid, kFwdThreads, smem, stream>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    g_last_cuda_error = (int)e;
    return REHR_CUDA_ERROR;
  }
  if (ksplit > 1) {
    if (rc)
      conv_splitk_finish_kernel<true><<<dim3(total_tiles, BN / 16), 128, 0, stream>>>(p);
    else
      conv_splitk_finish_kernel<false><<<dim3(total_tiles, BN / 16), 128, 0, stream>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess) {
      g_last_cuda_error = (int)e;
      return REHR_CUDA_ERROR;
    }
  }
  return REHR_OK;
}

// ------------------------------------------------------------------------------------------------
// Device: weight-gradient kernel.  D_g[(tap, cm), cn] += sum_vox X_tap[vox, cm] * Y[vox, cn]
// ------------------------------------------------------------------------------------------------
static constexpr int kMaxGroupsPerCta = 16;

struct alignas(64) WgradParams {
  CUtensorMap x_map[kMaxMaps];  // tapped operand (M side), box = (xa, box)
  CUtensorMap y_map;            // plain operand (N side), box = (ya, box)
  int2 taps[kMaxTaps];
  int num_taps;
  int box[4], tiles[4];  // voxel box (product BKV) over the Y grid
  int BKV;               // voxels per K block (128/64/32)
  int xa, ya;            // channel atoms (64/32/16) of X and Y
  int CM, CN;            // channels of X (M side) and Y (N side)
  int cmt;               // rows per tap inside a group: min(CM rounded to atom, 128)
  int tpg;               // taps per group (128 / cmt), 1 when CM >= 128
  int cm_tiles;          // ceil(CM / 128) when CM > 128 else 1
  int num_groups;        // total accumulator groups
  int gpc;               // groups per CTA item
  int group_sets;        // ceil(num_groups / gpc)
  int BN, n_tiles;       // N tile
  int splits;            // split-K factor
  int k_tiles;           // total voxel boxes
  int stages;
  int tmem_cols;
  float* ws;             // [split][group][128][CN]
  int* err;
};

__global__ void __launch_bounds__(kWgradThreads, 1) conv_wgrad_kernel(const __grid_constant__ WgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const uint32_t y_atom_bytes = (uint32_t)p.BKV * p.ya * 2u;
  const uint32_t y_bytes = y_atom_bytes * (uint32_t)(p.BN / p.ya);
  const uint32_t x_atom_bytes = (uint32_t)p.BKV * p.xa * 2u;
  const uint32_t x_group_bytes = (uint32_t)p.BKV * 128u * 2u;  // one accumulator group = 128 M rows
  const uint32_t stage_bytes = y_bytes + (uint32_t)p.gpc * x_group_bytes;
  uint8_t* tail = smem + (size_t)p.stages * stage_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_bar = full_bar + kMaxStages;
  uint64_t* done_bar = empty_bar + kMaxStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 2);

  if (warp == 0 && lane == 0) {
    for (int m = 0; m < kMaxMaps; ++m) tma_prefetch_desc(&p.x_map[m]);
    tma_prefetch_desc(&p.y_map);
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(&done_bar[0], 1);
    fence_mbar_init();
  } else if (warp == 1) {
    tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // work item of this CTA
  int item = blockIdx.x;
  const int split = item % p.splits;
  item /= p.splits;
  const int n_tile = item % p.n_tiles;
  const int gset = item / p.n_tiles;
  const int g0 = gset * p.gpc;
  const int ng = min(p.gpc, p.num_groups - g0);
  const int kt0 = (int)(((long long)p.k_tiles * split) / p.splits);
  const int kt1 = (int)(((long long)p.k_tiles * (split + 1)) / p.splits);

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      // bytes actually delivered per stage (only real taps / atoms are loaded)
      for (int kt = kt0; kt < kt1; ++kt) {
        int mt = kt;
        const int tw = mt % p.tiles[0];
        mt /= p.tiles[0];
        const int th = mt % p.tiles[1];
        mt /= p.tiles[1];
        const int td = mt % p.tiles[2];
        const int tn = mt / p.tiles[2];
        const int w0 = tw * p.box[0], h0 = th * p.box[1], d0 = td * p.box[2], n0 = tn * p.box[3];
        mbar_wait(&empty_bar[stage], phase ^ 1u, p.err, 11);
        uint8_t* sy = smem + (size_t)stage * stage_bytes;
        uint8_t* sx = sy + y_bytes;
        // count bytes first
        uint32_t bytes = y_bytes;
        for (int g = 0; g < ng; ++g) {
          const int gg = g0 + g;
          if (p.cm_tiles > 1) {
            bytes += x_atom_bytes * (uint32_t)(128 / p.xa);
          } else {
            const int t0 = gg * p.tpg;
            const int nt = min(p.tpg, p.num_taps - t0);
            bytes += x_atom_bytes * (uint32_t)(nt * (p.cmt / p.xa));
          }
        }
        mbar_arrive_expect_tx(&full_bar[stage], bytes);
        for (int a = 0; a < p.BN / p.ya; ++a)
          tma_load_5d(&p.y_map, &full_bar[stage], sy + (size_t)a * y_atom_bytes, n_tile * p.BN + a * p.ya, w0, h0, d0, n0);
        for (int g = 0; g < ng; ++g) {
          const int gg = g0 + g;
          uint8_t* sg = sx + (size_t)g * x_group_bytes;
          if (p.cm_tiles > 1) {
            const int tap = gg / p.cm_tiles, cmt_i = gg % p.cm_tiles;
            const int2 t = p.taps[tap];
            const int map_id = t.x & 0xff;
            const int dw = ((t.x >> 8) & 0xff) - 128, dh = ((t.x >> 16) & 0xff) - 128, dd = ((t.x >> 24) & 0xff) - 128;
            for (int a = 0; a < 128 / p.xa; ++a)
              tma_load_5d(&p.x_map[map_id], &full_bar[stage], sg + (size_t)a * x_atom_bytes, cmt_i * 128 + a * p.xa,
                          w0 + dw, h0 + dh, d0 + dd, n0);
          } else {
            const int t0 = gg * p.tpg;
            const int nt = min(p.tpg, p.num_taps - t0);
            const int apt = p.cmt / p.xa;  // atoms per tap
            for (int ti = 0; ti < nt; ++ti) {
              const int2 t = p.taps[t0 + ti];
              const int map_id = t.x & 0xff;
              const int dw = ((t.x >> 8) & 0xff) - 128, dh = ((t.x >> 16) & 0xff) - 128, dd = ((t.x >> 24) & 0xff) - 128;
              for (int a = 0; a < apt; ++a)
                tma_load_5d(&p.x_map[map_id], &full_bar[stage], sg + (size_t)(ti * apt + a) * x_atom_bytes, a * p.xa,
                            w0 + dw, h0 + dh, d0 + dd, n0);
            }
          }
        }
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = make_idesc_bf16(128, p.BN, 1, 1);
    const uint32_t x_row = (uint32_t)p.xa * 2u, y_row = (uint32_t)p.ya * 2u;
    const uint32_t x_layout = swizzle_layout_for_bytes((int)x_row), y_layout = swizzle_layout_for_bytes((int)y_row);
    // MN-major descriptors: LBO (bits 16..29 of the low word) = pitch between channel atoms, SBO = pitch between 8-voxel groups
    const uint32_t a_hi = (((8u * x_row) >> 4) & 0x3FFFu) | (1u << 14) | (x_layout << 29);
    const uint32_t b_hi = (((8u * y_row) >> 4) & 0x3FFFu) | (1u << 14) | (y_layout << 29);
    const uint32_t a_lbo = ((x_atom_bytes >> 4) & 0x3FFFu) << 16, b_lbo = ((y_atom_bytes >> 4) & 0x3FFFu) << 16;
    const uint32_t a_step = (16u * x_row) >> 4, b_step = (16u * y_row) >> 4;
    const uint32_t smem_lo = smem_u32(smem) >> 4, stage_lo = stage_bytes >> 4, y_lo = y_bytes >> 4, xg_lo = x_group_bytes >> 4;
    int stage = 0;
    uint32_t phase = 0;
    for (int kt = kt0; kt < kt1; ++kt) {
      mbar_wait(&full_bar[stage], phase, p.err, 12);
      tc_fence_after();
      const uint32_t sy_lo = smem_lo + (uint32_t)stage * stage_lo;
      if (elect_one()) {
        for (int g = 0; g < ng; ++g) {
          const uint32_t sg_lo = (sy_lo + y_lo + (uint32_t)g * xg_lo) | a_lbo;
          const uint32_t d_tmem = tmem_base + (uint32_t)(g * p.BN);
          if (p.BKV == 128) issue_kblock<8>(d_tmem, sg_lo, sy_lo | b_lbo, a_hi, b_hi, idesc, kt == kt0, a_step, b_step);
          else if (p.BKV == 64) issue_kblock<4>(d_tmem, sg_lo, sy_lo | b_lbo, a_hi, b_hi, idesc, kt == kt0, a_step, b_step);
          else issue_kblock<2>(d_tmem, sg_lo, sy_lo | b_lbo, a_hi, b_hi, idesc, kt == kt0, a_step, b_step);
        }
        umma_commit(&empty_bar[stage]);
        if (kt == kt1 - 1) umma_commit(&done_bar[0]);
      }
      __syncwarp();
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1u;
      }
    }
  } else {
    // epilogue: rows -> workspace [split][group][128][CN]
    const int q = warp & 3;
    const int row = q * 32 + lane;
    if (kt1 > kt0) {
      mbar_wait(&done_bar[0], 0, p.err, 13);
      tc_fence_after();
    }
    for (int g = 0; g < ng; ++g) {
      const int gg = g0 + g;
      float* dst = p.ws + (((long long)split * p.num_groups + gg) * 128 + row) * p.CN + n_tile * p.BN;
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(g * p.BN);
      for (int c0 = 0; c0 < p.BN; c0 += 16) {
        uint32_t v[16];
        if (kt1 > kt0) {
          tmem_ld16(taddr + (uint32_t)c0, v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = 0u;
        }
        const int cb = n_tile * p.BN + c0;
        if (cb + 16 <= p.CN && (p.CN & 3) == 0) {
#pragma unroll
          for (int i = 0; i < 16; i += 4)
            *reinterpret_cast<float4*>(dst + c0 + i) =
                make_float4(__uint_as_float(v[i]), __uint_as_float(v[i + 1]), __uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
        } else {
          for (int i = 0; i < 16; ++i)
            if (cb + i < p.CN) dst[c0 + i] = __uint_as_float(v[i]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// ws [split][group][128][CN] -> dw[cn*s_n + cm*s_m + widx*s_t]
struct WgradReduceParams {
  const float* ws;
  float* dw;
  int splits, num_groups, CN, CM, cm_tiles, tpg, cmt, num_taps;
  long long s_n, s_m, s_t;
  int accumulate;
  int widx[kMaxTaps];
};

__global__ void wgrad_reduce_serial_kernel(const WgradReduceParams p) {
  const long long total = (long long)p.num_groups * 128 * p.CN;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cn = (int)(i % p.CN);
    const long long gr = i / p.CN;
    const int m = (int)(gr % 128);
    const int g = (int)(gr / 128);
    int tap, cm;
    if (p.cm_tiles > 1) {
      tap = g / p.cm_tiles;
      cm = (g % p.cm_tiles) * 128 + m;
    } else {
      tap = g * p.tpg + m / p.cmt;
      cm = m % p.cmt;
      if (m / p.cmt >= p.tpg) continue;
    }
    if (tap >= p.num_taps || cm >= p.CM) continue;
    float acc = 0.f;
    for (int s = 0; s < p.splits; ++s) acc += p.ws[((long long)s * p.num_groups * 128 + gr) * p.CN + cn];
    float* d = p.dw + cn * p.s_n + cm * p.s_m + p.widx[tap] * p.s_t;
    *d = p.accumulate ? (*d + acc) : acc;
  }
}

// Long split lists (few accumulator groups => hundreds of split-K partials, e.g. the stride-2 32->64 layer):
// block = 32 (consecutive cn) x 8 (slices of the split list): the partial list of an output element is summed by 8 threads in
// an interleaved, fixed order and combined through shared memory (deterministic)
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const WgradReduceParams p) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const long long total = (long long)p.num_groups * 128 * p.CN;
  const long long i = (long long)blockIdx.x * 32 + lane;
  float acc = 0.f;
  bool live = i < total;
  int cn = 0, tap = 0, cm = 0;
  if (live) {
    cn = (int)(i % p.CN);
    const long long gr = i / p.CN;
    const int m = (int)(gr % 128);
    const int g = (int)(gr / 128);
    if (p.cm_tiles > 1) {
      tap = g / p.cm_tiles;
      cm = (g % p.cm_tiles) * 128 + m;
    } else {
      tap = g * p.tpg + m / p.cmt;
      cm = m % p.cmt;
      if (m / p.cmt >= p.tpg) live = false;
    }
    if (tap >= p.num_taps || cm >= p.CM) live = false;
    if (live)
      for (int s = slice; s < p.splits; s += 8) acc += p.ws[((long long)s * p.num_groups * 128 + gr) * p.CN + cn];
  }
  red[slice][lane] = acc;
  __syncthreads();
  if (slice == 0 && live) {
    float t = 0.f;
#pragma unroll
    for (int s = 0; s < 8; ++s) t += red[s][lane];
    float* d = p.dw + cn * p.s_n + cm * p.s_m + p.widx[tap] * p.s_t;
    *d = p.accumulate ? (*d + t) : t;
  }
}

// PyTorch-layout outputs (s_t == 1, s_m == T: the T taps of one (cn, cm) pair are contiguous): block = 32 cn x 8 cm.  Reads stay
// coalesced over cn; the sums go through a shared-memory tile so that every cn row is written as one contiguous run of 8*T floats
// (the element-per-thread kernels above write 4 bytes per 32-byte sector).  Fixed summation order -> deterministic.
__global__ void __launch_bounds__(256) wgrad_reduce_tiled_kernel(const WgradReduceParams p, int T) {
  extern __shared__ float sm[];  // [32][8*T + 1], then T present-flags
  const int rowlen = 8 * T + 1;
  int* present = reinterpret_cast<int*>(sm + 32 * rowlen);
  const int lane = threadIdx.x & 31, wy = threadIdx.x >> 5;
  for (int t = threadIdx.x; t < T; t += 256) present[t] = 0;
  __syncthreads();
  for (int j = threadIdx.x; j < p.num_taps; j += 256) present[p.widx[j]] = 1;
  const int cn = blockIdx.x * 32 + lane;
  const int cm = blockIdx.y * 8 + wy;
  if (cn < p.CN && cm < p.CM) {
    const long long split_stride = (long long)p.num_groups * 128 * p.CN;
#pragma unroll 3
    for (int j = 0; j < p.num_taps; ++j) {
      long long gr;
      if (p.cm_tiles > 1) gr = ((long long)j * p.cm_tiles + cm / 128) * 128 + (cm % 128);
      else gr = (long long)(j / p.tpg) * 128 + (j % p.tpg) * p.cmt + cm;
      const float* src = p.ws + gr * p.CN + cn;
      // four independent partial sums: the loads of a tap's split list are in flight together (the chain was latency bound)
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      int sp = 0;
      for (; sp + 4 <= p.splits; sp += 4) {
        const float v0 = src[(sp + 0) * split_stride], v1 = src[(sp + 1) * split_stride];
        const float v2 = src[(sp + 2) * split_stride], v3 = src[(sp + 3) * split_stride];
        a0 += v0; a1 += v1; a2 += v2; a3 += v3;
      }
      for (; sp < p.splits; ++sp) a0 += src[sp * split_stride];
      sm[lane * rowlen + wy * T + p.widx[j]] = (a0 + a1) + (a2 + a3);
    }
  }
  __syncthreads();
  const int cm0 = blockIdx.y * 8;
  for (int idx = threadIdx.x; idx < 32 * 8 * T; idx += 256) {
    const int cnl = idx / (8 * T), off = idx - cnl * (8 * T);
    const int cml = off / T, t = off - cml * T;
    const int c_n = blockIdx.x * 32 + cnl;
    if (c_n >= p.CN || cm0 + cml >= p.CM || !present[t]) continue;
    float* d = p.dw + c_n * p.s_n + (long long)cm0 * T + off;
    const float v = sm[cnl * rowlen + off];
    *d = p.accumulate ? (*d + v) : v;
  }
}

struct WgradPlan {
  WgradParams p;
  size_t ws_bytes;
  size_t smem;
  int grid;
};

static int plan_wgrad(const TapPlan& plan, const rehr_tensor& X, const rehr_tensor& Y, WgradPlan* out, bool encode) {
  WgradParams& p = out->p;
  memset(&p, 0, sizeof(p));
  const int CM = X.c, CN = Y.c;
  const int xa = chunk_for_channels(CM), ya = chunk_for_channels(CN);
  if (xa == 0 || ya == 0) return REHR_UNSUPPORTED;
  if (X.ld % 8 != 0 || Y.ld % 8 != 0) return REHR_BAD_ALIGNMENT;
  p.xa = xa;
  p.ya = ya;
  p.CM = CM;
  p.CN = CN;
  p.num_taps = plan.num_taps;
  if (CM <= 128 && 128 % CM != 0) return REHR_UNSUPPORTED;
  if (CM > 128) {
    p.cm_tiles = (CM + 127) / 128;
    p.cmt = 128;
    p.tpg = 1;
    p.num_groups = plan.num_taps * p.cm_tiles;
  } else {
    p.cm_tiles = 1;
    p.cmt = CM;  // multiple of xa
    p.tpg = 128 / CM;
    p.num_groups = (plan.num_taps + p.tpg - 1) / p.tpg;
  }
  // N tiling (multiple of ya, <= 256)
  {
    const int units = (CN + ya - 1) / ya;
    const int max_units = 256 / ya;
    p.n_tiles = (units + max_units - 1) / max_units;
    p.BN = ((units + p.n_tiles - 1) / p.n_tiles) * ya;
  }
  p.gpc = std::min(std::min(512 / p.BN, kMaxGroupsPerCta), p.num_groups);
  // shared memory: choose the largest voxel block that still leaves >= 2 stages
  const size_t tailb = (2 * kMaxStages + 2) * 8 + 64;
  const size_t budget = smem_budget() - 1024 - tailb;
  int BKV = 128;
  for (;;) {
    size_t sb = (size_t)BKV * 2 * (p.BN + (size_t)p.gpc * 128);
    if (budget / sb >= 2 || BKV == 32) break;
    BKV >>= 1;
  }
  while ((size_t)BKV * 2 * (p.BN + (size_t)p.gpc * 128) * 2 > budget && p.gpc > 1) p.gpc--;
  const size_t stage_bytes = (size_t)BKV * 2 * (p.BN + (size_t)p.gpc * 128);
  if (stage_bytes * 2 > budget) return REHR_UNSUPPORTED;
  p.BKV = BKV;
  p.stages = (int)std::min<size_t>(kMaxStages, budget / stage_bytes);
  p.group_sets = (p.num_groups + p.gpc - 1) / p.gpc;
  int tc = 32;
  while (tc < p.gpc * p.BN) tc <<= 1;
  p.tmem_cols = tc;
  choose_box(Y.w, Y.h, Y.d, Y.n, BKV, p.box);
  const int ysz[4] = {Y.w, Y.h, Y.d, Y.n};
  p.k_tiles = 1;
  for (int a = 0; a < 4; ++a) {
    p.tiles[a] = (ysz[a] + p.box[a] - 1) / p.box[a];
    p.k_tiles *= p.tiles[a];
  }
  const int base_items = p.group_sets * p.n_tiles;
  int splits = std::max(1, (2 * sm_count()) / std::max(1, base_items));
  splits = std::min(splits, p.k_tiles);
  splits = std::min(splits, 1024);
  p.splits = splits;
  out->grid = base_items * splits;
  out->ws_bytes = (size_t)splits * p.num_groups * 128 * CN * sizeof(float);
  out->smem = 1024 + (size_t)p.stages * stage_bytes + tailb;
  for (int j = 0; j < plan.num_taps; ++j) {
    const Tap& t = plan.taps[j];
    if (t.dw < -128 || t.dw > 127 || t.dh < -128 || t.dh > 127 || t.dd < -128 || t.dd > 127) return REHR_UNSUPPORTED;
    p.taps[j].x = (t.map_id & 0xff) | ((t.dw + 128) << 8) | ((t.dh + 128) << 16) | ((t.dd + 128) << 24);
    p.taps[j].y = t.widx;
  }
  if (!encode) return REHR_OK;

  const long long pw = X.ld, ph = (long long)X.w * X.ld, pd = (long long)X.h * ph, pn = (long long)X.d * pd;
  const long long base_pitch[3] = {pw, ph, pd};
  const int isz[3] = {X.w, X.h, X.d};
  for (int m = 0; m < kMaxMaps; ++m) {
    const int mm = m < plan.num_maps ? m : 0;
    int ext[4];
    long long pitch[4];
    long long off = 0;
    for (int a = 0; a < 3; ++a) {
      const int s = plan.map_s[mm][a], r = plan.map_r[mm][a];
      ext[a] = (isz[a] - r + s - 1) / s;
      pitch[a] = base_pitch[a] * s;
      off += (long long)r * base_pitch[a];
    }
    ext[3] = X.n;
    pitch[3] = pn;
    int rc = encode_act_map(&p.x_map[m], reinterpret_cast<const __nv_bfloat16*>(X.ptr) + off, CM, ext, pitch, xa, p.box);
    if (rc != REHR_OK) return rc;
  }
  {
    int ext[4] = {Y.w, Y.h, Y.d, Y.n};
    long long pitch[4] = {Y.ld, (long long)Y.w * Y.ld, (long long)Y.h * Y.w * Y.ld, (long long)Y.d * Y.h * Y.w * Y.ld};
    int rc = encode_act_map(&p.y_map, Y.ptr, CN, ext, pitch, ya, p.box);
    if (rc != REHR_OK) return rc;
  }
  return REHR_OK;
}

size_t tapped_wgrad_workspace(const TapPlan& plan, const rehr_tensor& X, const rehr_tensor& Y) {
  WgradPlan wp;
  if (plan_wgrad(plan, X, Y, &wp, false) != REHR_OK) return 0;
  return wp.ws_bytes;
}

// dw[cn*s_n + cm*s_m + widx*s_t] (+)= sum_o X_tap[o, cm] * Y[o, cn]
int launch_tapped_wgrad(const TapPlan& plan, const rehr_tensor& X, const rehr_tensor& Y, float* dw, long long s_n,
                        long long s_m, long long s_t, int accumulate, void* ws, size_t ws_bytes, cudaStream_t stream) {
  WgradPlan wp;
  int rc = plan_wgrad(plan, X, Y, &wp, true);
  if (rc != REHR_OK) return rc;
  if (ws_bytes < wp.ws_bytes || ws == nullptr) return REHR_WORKSPACE;
  wp.p.ws = reinterpret_cast<float*>(ws);
  wp.p.err = nullptr;
  REHR_SET_MAX_SMEM_ONCE(conv_wgrad_kernel, 227 * 1024);
  conv_wgrad_kernel<<<wp.grid, kWgradThreads, wp.smem, stream>>>(wp.p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    g_last_cuda_error = (int)e;
    return REHR_CUDA_ERROR;
  }
  WgradReduceParams r;
  r.ws = wp.p.ws;
  r.dw = dw;
  r.splits = wp.p.splits;
  r.num_groups = wp.p.num_groups;
  r.CN = wp.p.CN;
  r.CM = wp.p.CM;
  r.cm_tiles = wp.p.cm_tiles;
  r.tpg = wp.p.tpg;
  r.cmt = wp.p.cmt;
  r.num_taps = plan.num_taps;
  r.s_n = s_n;
  r.s_m = s_m;
  r.s_t = s_t;
  r.accumulate = accumulate;
  for (int j = 0; j < plan.num_taps; ++j) r.widx[j] = plan.taps[j].widx;
  const long long total = (long long)r.num_groups * 128 * r.CN;
  const int T = (int)s_m;
  bool tiled = s_t == 1 && T >= plan.num_taps && T <= 32 && r.splits < 24 && (r.cm_tiles > 1 || r.cmt >= r.CM);
  for (int j = 0; j < plan.num_taps && tiled; ++j) tiled = r.widx[j] >= 0 && r.widx[j] < T;
  if (tiled) {
    const size_t smem = (size_t)32 * (8 * T + 1) * sizeof(float) + (size_t)T * sizeof(int);
    wgrad_reduce_tiled_kernel<<<dim3((r.CN + 31) / 32, (r.CM + 7) / 8), 256, smem, stream>>>(r, T);
  } else if (r.splits >= 24) {
    wgrad_reduce_kernel<<<(int)((total + 31) / 32), 256, 0, stream>>>(r);
  } else {
    const int blocks = (int)std::min<long long>((total + 255) / 256, 148 * 8);
    wgrad_reduce_serial_kernel<<<blocks, 256, 0, stream>>>(r);
  }
  e = cudaGetLastError();
  if (e != cudaSuccess) {
    g_last_cuda_error = (int)e;
    return REHR_CUDA_ERROR;
  }
  return REHR_OK;
}

// ------------------------------------------------------------------------------------------------
// Weight packing: f32 src[r*sr + c*sc + t*st] -> bf16 dst[r][t][c]
// ------------------------------------------------------------------------------------------------
__global__ void pack_weight_kernel(const float* __restrict__ src, unsigned short* __restrict__ dst, int R, int C, int T,
                                   long long sr, long long sc, long long st, int f16) {
  const long long total = (long long)R * T * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const long long rt = i / C;
    const int t = (int)(rt % T);
    const int r = (int)(rt / T);
    dst[i] = pack16(src[r * sr + c * sc + t * st], f16);
  }
}

// st == 1 (the T taps of one (r, c) pair are contiguous in src): block = (r, 64 consecutive c); the 64 runs of T floats are
// read coalesced into shared memory and written back transposed as 64 consecutive bf16 per tap.
static constexpr int kPackC = 64;
__global__ void __launch_bounds__(256) pack_weight_runs_kernel(const float* __restrict__ src, unsigned short* __restrict__ dst, int R,
                                                               int C, int T, long long sr, long long sc, int f16) {
  extern __shared__ float tile[];  // [kPackC][T + 1]
  const int r = blockIdx.y, c0 = blockIdx.x * kPackC;
  const int nc = min(kPackC, C - c0);
  for (int i = threadIdx.x; i < nc * T; i += 256) {
    const int cl = i / T, t = i % T;
    tile[cl * (T + 1) + t] = src[r * sr + (long long)(c0 + cl) * sc + t];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nc * T; i += 256) {
    const int t = i / nc, cl = i % nc;
    dst[((long long)r * T + t) * C + c0 + cl] = pack16(tile[cl * (T + 1) + t], f16);
  }
}

int launch_pack_weight(const float* src, void* dst, int R, int C, int T, long long sr, long long sc, long long st,
                       cudaStream_t stream, int f16) {
  const long long total = (long long)R * T * C;
  if (total == 0) return REHR_OK;
  if (pack_recording()) {
    PackJob j{};
    j.src = src; j.dst = dst; j.kind = 0; j.f16 = f16;
    j.R = R; j.C = C; j.T = T; j.sr = sr; j.sc = sc; j.st = st;
    return pack_record(j);
  }
  if (st == 1 && T <= 343 && R <= 65535) {
    dim3 grid((C + kPackC - 1) / kPackC, R);
    const size_t smem = (size_t)kPackC * (T + 1) * sizeof(float);
    if (smem > 48 * 1024) REHR_SET_MAX_SMEM_ONCE(pack_weight_runs_kernel, 96 * 1024);
    pack_weight_runs_kernel<<<grid, 256, smem, stream>>>(src, reinterpret_cast<unsigned short*>(dst), R, C, T, sr, sc, f16);
  } else {
    const int blocks = (int)std::min<long long>((total + 255) / 256, 148 * 16);
    pack_weight_kernel<<<blocks, 256, 0, stream>>>(src, reinterpret_cast<unsigned short*>(dst), R, C, T, sr, sc, st, f16);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    g_last_cuda_error = (int)e;
    return REHR_CUDA_ERROR;
  }
  return REHR_OK;
}

}  // namespace rehr
