// "Marching" convolution kernel for sm_100a: k = 3x3x3, stride 1, pad 1, few channels (the layers that hold
// 3/4 of the nnU-Net FLOPs: 32->32, 64->32, 64->64, 128->64 at 128^3 / 64^3 -- SURVEY.md section 7.3).
//
// Why a second kernel: with Cout = 32..64 the generic tapped GEMM (conv_engine.cu) re-fetches every input voxel
// 27 times from L2 (one TMA box per tap) and is L2->SMEM bound at ~10 % of tensor peak.  Here
//   * a CTA owns a column of output voxels: a 16(h) x 8(w) in-plane tile, marched along d for a segment of planes;
//   * each input plane (18 x 10 halo'd voxels x Cin, ONE TMA box per 64-channel chunk) is loaded once into a shared
//     memory ring; the 9 in-plane taps (kh,kw) are NOT re-loaded: they are UMMA descriptor offsets into that tile
//     (row shift kh*10+kw, 8-row groups 10 rows apart).  Verified on B200: swizzled K-major descriptors use absolute
//     smem address bits, so arbitrary row shifts are legal (profiles/r01_umma_shifted_descriptor_probe.log);
//   * the 3 depth taps are fused into ONE tcgen05.mma: B = [W(kd=2) | W(kd=1) | W(kd=0)] (N = 3*Ct) and the
//     accumulators of output planes p-1, p, p+1 sit in adjacent TMEM column slots, so input plane p is read from
//     shared memory once per (kh,kw,k-step) instead of three times.  This lifts the A-operand SMEM read bound
//     (128x16 bf16 = 4 KB per MMA at 128 B/clk = 32 clk) above the MMA time (N/2 = 48 clk for Ct = 32);
//   * all 27*Cin*Ct weights stay resident in shared memory (Ct = output-channel tile chosen to fit);
//   * epilogue warps drain one finished plane at a time (bias, InstanceNorm partial sums, activation, bf16 store),
//     re-zero the TMEM slot (every MMA accumulates; there is no per-column "overwrite" flag) and hand it back.
// The same kernel is the input-gradient of those layers (weights packed transposed + tap-flipped).
//
// Reference call sites replaced: ConvDropoutNormReLU.conv of the full-resolution nnU-Net stages (built at
// models/seg_model.py:174-191), sr_head.0 (models/seg_model.py:197), FLAVR Conv3DSimple k3 (resnet_3D.py:19-33).
#include "engine.h"
#include "ptx.cuh"
#include "reduce.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

namespace rehr {

int encode_tiled_bf16(CUtensorMap* m, const void* base, int rank, const unsigned long long* gdim,
                      const unsigned long long* gstride_bytes, const unsigned* box, int swizzle_bytes);

static constexpr int kMarchThreads = 192;  // warp0 TMA, warp1 MMA (+TMEM alloc), warps 2..5 epilogue
static constexpr int kTileH = 16, kTileW = 8;
// kernel size KS (3 or 5, cubic, stride 1, pad (KS-1)/2): halo'd input tile of (16 + KS - 1) x (8 + KS - 1) voxels
template <int KS>
struct MarchGeo {
  static constexpr int R = (KS - 1) / 2;
  static constexpr int kHaloH = kTileH + KS - 1, kHaloW = kTileW + KS - 1, kHaloRows = kHaloH * kHaloW;  // k3: 18 x 10 = 180
};
static constexpr int kMaxRing = 8;
static constexpr int kMaxSlots = 16;

struct alignas(64) MarchParams {
  CUtensorMap x_map;  // 5-D NDHWC, box (BK, 10, 18, 1, 1)
  CUtensorMap w_map;  // 2-D [n_ct*9*chunks*3Ct rows][BK], box (BK, 3Ct)
  int N, D, H, W, Cin, Cout;
  int ks;  // 3 or 5 (in-plane extent; the depth extent is 1 for the planar k(1,3,3) layers, see kd_off)
  // planar layers (k = (1,3,3), pad (0,1,1): the thick-slice stages of anisotropic nnU-Net plans) run as the centre depth tap
  // only (kd_lo = kd_hi = R) and store just that tap: wrows = weight rows per (kh,kw,chunk) tile (= Ct instead of KS*Ct),
  // kd_off = index of the first stored depth tap (R instead of 0)
  int wrows, kd_off;
  // tap-index ranges actually present (the rest of the packed weights are zero and are skipped): whole kernel by default; the
  // parity classes of a stride-2 input gradient use 1 or 2 of the 3 taps per dimension (see rehr_conv3d_march_s2dgrad)
  int kd_lo, kd_hi, kh_lo, kh_hi, kw_lo, kw_hi;
  // output addressing: element offset = n*o_pn + d*o_pd + h*o_ph + w*o_pw (dense NDHWC by default; a parity class of a
  // larger tensor otherwise) and the extents that really exist (<= D, H, W)
  long long o_pn, o_pd, o_ph, o_pw;
  int OD, OH, OW;
  int Ct, n_ct, BK, chunks;
  int tiles_h, tiles_w, Ds, n_seg;
  int ring, slots;
  int total_items, items_per_ct;
  uint32_t w_bytes, plane_bytes, chunk_stride, slot_stride, wtile_bytes;
  void* out;
  int out_f32;
  int out_f16;  // 16-bit output format (rehr_dtype of y) when !out_f32
  int in_f16;   // MMA operand format: of x and of the packed weights (one format per tcgen05.mma)
  RangeSlot* range;  // fp16 saturation record of the stored values (rehr_range_sink), null = not checked
  long long out_ld;
  const float* bias;
  int act;
  float slope;
  float* stats;  // [N][tiles_per_sample][Cout][2] or null
  int* err;
  long long* prof;  // development only: per-role cycle counters of CTA 0 (env REHR_MARCH_PROF)
  int debug;  // development only (env REHR_MARCH_DEBUG): bit0 skip input TMA, bit1 skip epilogue body, bit2 skip MMAs
};

__device__ __forceinline__ float march_act(float v, int act, float slope) {
  if (act == REHR_ACT_RELU) return v > 0.f ? v : 0.f;
  if (act == REHR_ACT_LRELU) return v > 0.f ? v : v * slope;
  return v;
}

struct ItemCoord {
  int ct, n, seg, th, tw;
};
__device__ __forceinline__ ItemCoord decode_item(const MarchParams& p, int item) {
  ItemCoord c;
  c.ct = item / p.items_per_ct;
  int r = item - c.ct * p.items_per_ct;
  c.tw = r % p.tiles_w;
  r /= p.tiles_w;
  c.th = r % p.tiles_h;
  r /= p.tiles_h;
  c.seg = r % p.n_seg;
  c.n = r / p.n_seg;
  return c;
}

__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}

// BKT = channels per K chunk (16 / 32 / 64 -> 32 / 64 / 128 B swizzled rows), CHUNKS = Cin / BKT, CT = output-channel
// tile (epilogue keeps CT running column sums per thread in registers).  Compile-time so that
// the MMA issue sequence of one input plane (9 * CHUNKS * BKT/16 instructions) is fully unrolled with constant
// descriptor increments: a single thread must issue one tcgen05.mma every ~50 clk (tools/umma_rate2.cu measures
// 40 clk/MMA for this code shape vs 120-280 clk/MMA with run-time descriptor arithmetic).
// REHR_MARCH_MAXNREG (build-time, default = no cap): register cap of the kernel.  A 128-register build lets two blocks of an
// InstanceNorm pass become resident next to a conv CTA (tools/overlap_probe.py: 55 % of a co-scheduled pass hides behind a
// forward conv instead of 12 %) but costs the conv itself 5 % (spilled column sums); measured on the C1 step: a net loss.
// The kernel carries both .maxntid and .maxnreg: ptxas allocates registers differently with the explicit cap than without it
// (94 instead of 80 for the 16-channel tile), and the kernels were measured that way.  nvcc accepts __launch_bounds__ together
// with __maxnreg__ only when an argument depends on a template parameter, hence the KS term.
#ifndef REHR_MARCH_MAXNREG
#define REHR_MARCH_MAXNREG 255
#endif
// RC: the fp16 saturation check of the stored values (p.range != null) is compiled in; the unchecked instantiation is the kernel
// without it (with a run-time test instead, this register-bound epilogue ran up to a quarter slower with the check off).
template <int BKT, int CHUNKS, int CT, int KS, bool RC>
__global__ void __launch_bounds__(kMarchThreads) __maxnreg__(KS > 0 ? REHR_MARCH_MAXNREG : 0) conv_march_kernel(const __grid_constant__ MarchParams p) {
  constexpr int R = MarchGeo<KS>::R;
  constexpr int kHaloW = MarchGeo<KS>::kHaloW;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* s_w = smem;                                   // resident weights
  uint8_t* s_ring = smem + ((p.w_bytes + 1023u) & ~1023u);  // input plane ring
  uint8_t* tail = s_ring + (size_t)p.ring * p.slot_stride;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);  // [ring]
  uint64_t* empty_bar = full_bar + kMaxRing;               // [ring]
  uint64_t* tfull_bar = empty_bar + kMaxRing;              // [slots]
  uint64_t* tempty_bar = tfull_bar + kMaxSlots;            // [slots]
  uint64_t* wfull_bar = tempty_bar + kMaxSlots;            // [1]
  uint64_t* wfree_bar = wfull_bar + 1;                     // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wfree_bar + 1);
  float* part = reinterpret_cast<float*>(tmem_slot + 4);   // [4 warps][2][64]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kSlots = (512 / CT) < kMaxSlots ? (512 / CT) : kMaxSlots;  // power of two
  constexpr int kSlotMask = kSlots - 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.x_map);
    tma_prefetch_desc(&p.w_map);
    for (int i = 0; i < p.ring; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < p.slots; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 4);
    }
    mbar_init(wfull_bar, 1);
    mbar_init(wfree_bar, 1);
    fence_mbar_init();
  } else if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t rowb = (uint32_t)p.BK * 2u;

  if (warp == 0) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int cur_ct = -1;
      uint32_t wfree_phase = 0;
      for (int item = blockIdx.x; item < p.total_items; item += gridDim.x) {
        const ItemCoord c = decode_item(p, item);
        if (c.ct != cur_ct) {
          if (cur_ct >= 0) {  // wait until every MMA that reads the old weights has retired
            mbar_wait(wfree_bar, wfree_phase, p.err, 21);
            wfree_phase ^= 1u;
          }
          cur_ct = c.ct;
          mbar_arrive_expect_tx(wfull_bar, p.w_bytes);
          const int tiles = KS * KS * p.chunks;
          for (int t = 0; t < tiles; ++t)
            tma_load_2d(&p.w_map, wfull_bar, s_w + (size_t)t * p.wtile_bytes, 0, (c.ct * tiles + t) * p.wrows);
        }
        const int d0 = c.seg * p.Ds, d1 = min(p.D, d0 + p.Ds);
        const int pa = max(d0 + p.kd_lo - R, 0), pb = min(d1 - 1 + p.kd_hi - R, p.D - 1);
        const int h0 = c.th * kTileH - R, w0 = c.tw * kTileW - R;
        for (int pl = pa; pl <= pb; ++pl) {
          const long long tp0 = clock64();
          mbar_wait(&empty_bar[stage], phase ^ 1u, p.err, 22);
          if (p.prof && blockIdx.x == 0) { p.prof[0] += clock64() - tp0; p.prof[1] += 1; }
          if (p.debug & 1) {
            mbar_arrive(&full_bar[stage]);
          } else {
            mbar_arrive_expect_tx(&full_bar[stage], p.plane_bytes);
            uint8_t* dst = s_ring + (size_t)stage * p.slot_stride;
            for (int ch = 0; ch < p.chunks; ++ch)
              tma_load_5d(&p.x_map, &full_bar[stage], dst + (size_t)ch * p.chunk_stride, ch * p.BK, w0, h0, pl, c.n);
          }
          if (++stage == p.ring) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer ==============================
    // The whole warp runs the (warp-uniform) control flow and barrier waits; one elected lane issues the MMAs.
    constexpr uint32_t kRowB = BKT * 2;
    constexpr int kSteps = BKT / 16;
    constexpr uint32_t kLayout = kRowB == 128 ? 2u : (kRowB == 64 ? 4u : 6u);
    // high words of the K-major descriptors: SBO (bits 32..45), version 1 (bit 46), swizzle mode (bits 61..63)
    constexpr uint32_t kAHi = ((kHaloW * kRowB) >> 4) | (1u << 14) | (kLayout << 29);
    constexpr uint32_t kBHi = ((8u * kRowB) >> 4) | (1u << 14) | (kLayout << 29);
    const uint32_t sw_lo = smem_u32(s_w) >> 4, sring_lo = smem_u32(s_ring) >> 4;
    const uint32_t slot_lo = p.slot_stride >> 4, chunk_lo = p.chunk_stride >> 4, wtile_lo = p.wtile_bytes >> 4;
    int stage = 0;
    uint32_t phase = 0;
    int cur_ct = -1;
    uint32_t wfull_phase = 0;
    uint32_t tempty_par = 0;  // bit s = parity to wait for on tempty_bar[s]
    for (int item = blockIdx.x; item < p.total_items; item += gridDim.x) {
      const ItemCoord c = decode_item(p, item);
      if (c.ct != cur_ct) {
        cur_ct = c.ct;
        mbar_wait(wfull_bar, wfull_phase, p.err, 31);
        wfull_phase ^= 1u;
        tc_fence_after();
      }
      const int d0 = c.seg * p.Ds, d1 = min(p.D, d0 + p.Ds);
      const int pa = max(d0 + p.kd_lo - R, 0), pb = min(d1 - 1 + p.kd_hi - R, p.D - 1);
      int next_open = d0;
      for (int pl = pa; pl <= pb; ++pl) {
        // input plane pl feeds output plane q through depth tap kd = pl - q + R, kd in [kd_lo, kd_hi]
        const int qa = max(pl - p.kd_hi + R, d0), qb = min(pl - p.kd_lo + R, d1 - 1);
        const long long tm0 = clock64();
        while (next_open <= qb) {  // first touch of an output plane's TMEM slot: wait until it was drained + zeroed
          const int s = (next_open - d0) & kSlotMask;
          mbar_wait(&tempty_bar[s], (tempty_par >> s) & 1u, p.err, 32);
          tempty_par ^= 1u << s;
          ++next_open;
        }
        const long long tm1 = clock64();
        mbar_wait(&full_bar[stage], phase, p.err, 33);
        tc_fence_after();
        const long long tm2 = clock64();
        const uint32_t a_lo = sring_lo + (uint32_t)stage * slot_lo;
        // contiguous TMEM slot runs covering output planes qa..qb (one run unless the slot ring wraps)
        int ra = qa;
        while (ra <= qb) {
          int rb = ra;
          while (rb < qb && ((rb + 1 - d0) & kSlotMask) != 0) ++rb;
          const uint32_t idesc = make_idesc_16(128, (rb - ra + 1) * CT, 0, 0, p.in_f16);
          const uint32_t b_lo = sw_lo + (((uint32_t)((ra - pl + R - p.kd_off) * CT) * kRowB) >> 4);
          const uint32_t d_tmem = tmem_base + (uint32_t)(((ra - d0) & kSlotMask) * CT);
          if (!(p.debug & 4) && elect_one_sync()) {
#pragma unroll
            for (int khw = 0; khw < KS * KS; ++khw) {
              if (khw / KS < p.kh_lo || khw / KS > p.kh_hi || khw % KS < p.kw_lo || khw % KS > p.kw_hi) continue;  // zero taps
#pragma unroll
              for (int ch = 0; ch < CHUNKS; ++ch) {
                const uint32_t a_t = a_lo + (uint32_t)((((khw / KS) * kHaloW + (khw % KS)) * kRowB) >> 4) + (uint32_t)ch * chunk_lo;
                const uint32_t b_t = b_lo + (uint32_t)(khw * CHUNKS + ch) * wtile_lo;
#pragma unroll
                for (int k = 0; k < kSteps; ++k) {
                  const uint64_t ad = ((uint64_t)kAHi << 32) | (uint64_t)(a_t + 2u * k);
                  const uint64_t bd = ((uint64_t)kBHi << 32) | (uint64_t)(b_t + 2u * k);
                  umma_bf16(d_tmem, ad, bd, idesc, 1u);
                }
              }
            }
          }
          __syncwarp();
          ra = rb + 1;
        }
        if (elect_one_sync()) {
          umma_commit(&empty_bar[stage]);
          // finished output planes
          // output plane q is complete once its last contributing input plane q + kd_hi - R has been issued
          const int qdone = pl - p.kd_hi + R;
          if (qdone >= d0 && qdone <= d1 - 1) umma_commit(&tfull_bar[(qdone - d0) & kSlotMask]);
          if (pl == pb) {
            for (int q = max(qdone + 1, d0); q <= d1 - 1; ++q) umma_commit(&tfull_bar[(q - d0) & kSlotMask]);
          }
        }
        __syncwarp();
        if (p.prof && blockIdx.x == 0 && lane == 0) {
          const long long tm3 = clock64();
          p.prof[4] += tm1 - tm0; p.prof[5] += tm2 - tm1; p.prof[6] += tm3 - tm2; p.prof[7] += 1;
        }
        if (++stage == p.ring) {
          stage = 0;
          phase ^= 1u;
        }
      }
      // tell the producer the weights may be replaced (only signalled when the next item needs other weights)
      const int nitem = item + gridDim.x;
      if (nitem < p.total_items && nitem / p.items_per_ct != c.ct) {
        if (elect_one_sync()) umma_commit(wfree_bar);
        __syncwarp();
      }
    }
  } else {
    // ============================== epilogue (warps 2..5) ==============================
    const int q4 = warp & 3;
    const int row = q4 * 32 + lane;
    const int hl = row >> 3, wl = row & 7;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q4 * 32) << 16);
    // zero the whole accumulator space once; afterwards every drained slot is re-zeroed
    {
      uint32_t z[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) z[i] = 0u;
      for (int c0 = 0; c0 < 512; c0 += 16) tmem_st16(lane_addr + (uint32_t)c0, z);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0)
        for (int s = 0; s < p.slots; ++s) mbar_arrive(&tempty_bar[s]);
    }
    uint32_t tfull_par = 0;
    const int et = threadIdx.x - 64;
    constexpr int kW = CT >= 32 ? 32 : 16;  // columns per TMEM round trip
    for (int item = blockIdx.x; item < p.total_items; item += gridDim.x) {
      const ItemCoord c = decode_item(p, item);
      const int d0 = c.seg * p.Ds, d1 = min(p.D, d0 + p.Ds);
      const int oh = c.th * kTileH + hl, ow = c.tw * kTileW + wl;
      const bool valid_hw = oh < p.OH && ow < p.OW;
      const int cbase = c.ct * CT;
      // per-thread running column sums of this item (this thread's output row, all planes of the segment)
      float s1[CT], s2[CT];
#pragma unroll
      for (int i = 0; i < CT; ++i) s1[i] = s2[i] = 0.f;
      for (int q = d0; q < d1; ++q) {
        const int s = (q - d0) & kSlotMask;
        const long long te0 = clock64();
        mbar_wait(&tfull_bar[s], (tfull_par >> s) & 1u, p.err, 41);
        tfull_par ^= 1u << s;
        tc_fence_after();
        const long long te1 = clock64();
        const uint32_t taddr = lane_addr + (uint32_t)(s * CT);
        const bool valid = valid_hw && q < p.OD;
        const long long obase = (long long)c.n * p.o_pn + (long long)q * p.o_pd + (long long)oh * p.o_ph + (long long)ow * p.o_pw;
#pragma unroll
        for (int c0 = 0; c0 < CT; c0 += kW) {
          if (p.debug & 2) break;
          uint32_t v[kW];
          if constexpr (kW == 32) tmem_ld32(taddr + (uint32_t)c0, v); else tmem_ld16(taddr + (uint32_t)c0, v);
          tmem_ld_wait();
          float f[kW];
#pragma unroll
          for (int i = 0; i < kW; ++i) f[i] = __uint_as_float(v[i]);
          const int nvalid = p.Cout - (cbase + c0);  // channels of this group that exist (Cout need not fill the tile)
          if (p.bias != nullptr) {
            if (nvalid >= kW) {
#pragma unroll
              for (int i = 0; i < kW; i += 4) {
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + cbase + c0 + i));
                f[i] += b4.x; f[i + 1] += b4.y; f[i + 2] += b4.z; f[i + 3] += b4.w;
              }
            } else {
#pragma unroll
              for (int i = 0; i < kW; ++i)
                if (i < nvalid) f[i] += __ldg(p.bias + cbase + c0 + i);
            }
          }
          if (p.stats != nullptr && valid) {
#pragma unroll
            for (int i = 0; i < kW; ++i) {
              s1[c0 + i] += f[i];
              s2[c0 + i] = fmaf(f[i], f[i], s2[c0 + i]);
            }
          }
          if (valid) {
#pragma unroll
            for (int i = 0; i < kW; ++i) f[i] = march_act(f[i], p.act, p.slope);
            const int cc = cbase + c0;
            if constexpr (RC) range_check<kW>(p.range, f, nvalid);
            if (nvalid < kW) {
              if (p.out_f32) {
                float* o = reinterpret_cast<float*>(p.out) + obase + cc;
#pragma unroll
                for (int i = 0; i < kW; ++i)
                  if (i < nvalid) o[i] = f[i];
              } else {
                unsigned short* o = reinterpret_cast<unsigned short*>(p.out) + obase + cc;
#pragma unroll
                for (int i = 0; i < kW; ++i)
                  if (i < nvalid) o[i] = pack16(f[i], p.out_f16);
              }
            } else if (p.out_f32) {
              float* o = reinterpret_cast<float*>(p.out) + obase + cc;
              if ((p.out_ld & 3) == 0) {
#pragma unroll
                for (int i = 0; i < kW; i += 4) *reinterpret_cast<float4*>(o + i) = make_float4(f[i], f[i + 1], f[i + 2], f[i + 3]);
              } else {
#pragma unroll
                for (int i = 0; i < kW; ++i) o[i] = f[i];
              }
            } else {
              unsigned short* o = reinterpret_cast<unsigned short*>(p.out) + obase + cc;
              if ((p.out_ld & 7) == 0) {
#pragma unroll
                for (int i = 0; i < kW; i += 8) {
                  uint4 u;
                  u.x = pack16x2(f[i], f[i + 1], p.out_f16);
                  u.y = pack16x2(f[i + 2], f[i + 3], p.out_f16);
                  u.z = pack16x2(f[i + 4], f[i + 5], p.out_f16);
                  u.w = pack16x2(f[i + 6], f[i + 7], p.out_f16);
                  *reinterpret_cast<uint4*>(o + i) = u;
                }
              } else {
#pragma unroll
                for (int i = 0; i < kW; ++i) o[i] = pack16(f[i], p.out_f16);
              }
            }
          }
          // re-zero the columns just read
          uint32_t z[kW];
#pragma unroll
          for (int i = 0; i < kW; ++i) z[i] = 0u;
          if constexpr (kW == 32) tmem_st32(taddr + (uint32_t)c0, z); else tmem_st16(taddr + (uint32_t)c0, z);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty_bar[s]);
        if (p.prof && blockIdx.x == 0 && threadIdx.x == 64) {
          p.prof[8] += te1 - te0; p.prof[9] += clock64() - te1; p.prof[10] += 1;
        }
      }
      if (p.stats != nullptr) {
        // cross-lane column totals (once per item) -> shared -> one partial per (item, channel)
#pragma unroll
        for (int c0 = 0; c0 < CT; c0 += 16) {
          float a1[16], a2[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            a1[i] = s1[c0 + i];
            a2[i] = s2[c0 + i];
          }
          warp_colsum16(a1, lane);
          warp_colsum16(a2, lane);
          if ((lane & 1) == 0) {
            const int col = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
            part[(q4 * 2 + 0) * 64 + c0 + col] = a1[0];
            part[(q4 * 2 + 1) * 64 + c0 + col] = a2[0];
          }
        }
        named_bar_sync(1, 128);
        if (et < CT && cbase + et < p.Cout) {
          float a = 0.f, b = 0.f;
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            a += part[(w * 2 + 0) * 64 + et];
            b += part[(w * 2 + 1) * 64 + et];
          }
          const int tiles_per_sample = p.n_seg * p.tiles_h * p.tiles_w;
          const int tile = (c.seg * p.tiles_h + c.th) * p.tiles_w + c.tw;
          float* dst = p.stats + (((long long)c.n * tiles_per_sample + tile) * p.Cout + cbase + et) * 2;
          dst[0] = a;
          dst[1] = b;
        }
        named_bar_sync(1, 128);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------
// Host planning
// ------------------------------------------------------------------------------------------------
static const size_t kMarchWeightBudget = 112 * 1024;

static inline int pad16(int c) { return (c + 15) / 16 * 16; }

// output-channel tile for a (cin, cout, ks) layer; 0 = not supported by the marching kernel
int march_ct(int cin, int cout, int ks, bool planar) {
  if (ks != 3 && ks != 5) return 0;
  if (planar && ks != 3) return 0;
  const int kdn = planar ? 1 : ks;  // stored depth taps
  if (cin % 16 != 0 || cout <= 0) return 0;
  if (cin != 16 && cin != 32 && cin != 64 && cin != 128) return 0;  // instantiated (BK, chunks) variants
  if (ks == 5 && cin != 16) return 0;                               // instantiated k5 variant: sr_head.2 (models/seg_model.py:199)
  const int cp = pad16(cout);
  for (int ct : {64, 32, 16}) {
    if (cp % ct != 0) continue;
    if (kdn * ct > 256) continue;  // kd-fused N and the weight TMA box are limited to 256 rows
    if (ks == 5 && ct != 16) continue;
    if ((size_t)kdn * ks * ks * cin * ct * 2 <= kMarchWeightBudget) return ct;
  }
  return 0;
}

struct MarchPlan {
  MarchParams p;
  size_t smem;
  int grid;
};

// barriers (full / empty ring, tfull / tempty slots, wfull, wfree), TMEM address, epilogue partials.  One more ring of barriers
// (8 * kMaxRing bytes) stays reserved: the plane-ring depths of the tuned layer shapes were measured with a tail of this size.
static size_t march_tail_bytes() { return (3 * kMaxRing + 2 * kMaxSlots + 2) * 8 + 16 + 4 * 2 * 64 * 4; }

static int plan_march(const rehr_tensor& x, const rehr_tensor& y, int ks_code, MarchPlan* out, int ds_override) {
  MarchParams& p = out->p;
  memset(&p, 0, sizeof(p));
  const bool planar = ks_code == 1;  // k(1,3,3)
  const int ks = planar ? 3 : ks_code;
  const int kdn = planar ? 1 : ks;
  const int ct = march_ct(x.c, y.c, ks, planar);
  if (ct == 0) return REHR_UNSUPPORTED;
  if (x.n != y.n || x.d != y.d || x.h != y.h || x.w != y.w) return REHR_BAD_SHAPE;
  p.N = x.n; p.D = x.d; p.H = x.h; p.W = x.w; p.Cin = x.c; p.Cout = y.c;
  p.ks = ks;
  p.kd_lo = p.kh_lo = p.kw_lo = 0;
  p.kd_hi = p.kh_hi = p.kw_hi = ks - 1;
  if (planar) p.kd_lo = p.kd_hi = (ks - 1) / 2;
  p.kd_off = planar ? (ks - 1) / 2 : 0;
  p.wrows = kdn * ct;
  p.OD = p.D; p.OH = p.H; p.OW = p.W;
  p.Ct = ct;
  p.n_ct = pad16(y.c) / ct;
  p.BK = std::min(x.c, 64);
  p.chunks = x.c / p.BK;
  p.tiles_h = (p.H + kTileH - 1) / kTileH;
  p.tiles_w = (p.W + kTileW - 1) / kTileW;
  p.slots = std::min(kMaxSlots, 512 / ct);
  const uint32_t rowb = p.BK * 2;
  const int halo_rows = (kTileH + ks - 1) * (kTileW + ks - 1);
  p.wtile_bytes = kdn * ct * rowb;
  p.w_bytes = ks * ks * p.chunks * p.wtile_bytes;
  p.chunk_stride = (halo_rows * rowb + 1023u) & ~1023u;
  p.slot_stride = p.chunks * p.chunk_stride;
  p.plane_bytes = p.chunks * halo_rows * rowb;
  const size_t fixed = 1024 + ((p.w_bytes + 1023u) & ~1023u) + march_tail_bytes();
  const size_t budget = smem_budget();
  if (fixed + 2 * (size_t)p.slot_stride > budget) return REHR_UNSUPPORTED;
  p.ring = (int)std::min<size_t>(kMaxRing, (budget - fixed) / p.slot_stride);
  out->smem = fixed + (size_t)p.ring * p.slot_stride;
  // depth segment: as long as possible while keeping >= ~6 work items per SM
  const int sms = sm_count();
  const long long cols = (long long)p.n_ct * p.N * p.tiles_h * p.tiles_w;
  int ds = p.D;
  while (ds > 8 && cols * ((p.D + ds - 1) / ds) < 6LL * sms) ds = (ds + 1) / 2;
  if (ds_override > 0) ds = ds_override;
  p.Ds = ds;
  p.n_seg = (p.D + ds - 1) / ds;
  p.items_per_ct = p.N * p.n_seg * p.tiles_h * p.tiles_w;
  p.total_items = p.items_per_ct * p.n_ct;
  out->grid = std::min(p.total_items, sms);
  return REHR_OK;
}

int march_stats_tiles(const rehr_tensor& x, const rehr_tensor& y, int ks) {
  MarchPlan pl;
  if (plan_march(x, y, ks, &pl, 0) != REHR_OK) return 0;
  return pl.p.n_seg * pl.p.tiles_h * pl.p.tiles_w;
}

static int dispatch_march(const MarchPlan& pl, cudaStream_t stream);

// Optional: restrict the taps and write one parity class of a larger tensor (stride-2 input gradients).
struct MarchExt {
  int lo[3], hi[3];            // tap ranges (d h w)
  long long pn, pd, ph, pw;    // output pitches in elements
  int OD, OH, OW;              // extents of the class that exist
};

int launch_march(const rehr_tensor& x, const void* w_march, const float* bias, const rehr_tensor& y, int ks_code, int y_is_f32, int act,
                 float slope, float* stats, cudaStream_t stream, const MarchExt* ext = nullptr) {
  MarchPlan pl;
  int rc = plan_march(x, y, ks_code, &pl, 0);
  if (rc != REHR_OK) return rc;
  MarchParams& p = pl.p;
  const int ks = p.ks;
  if (ext && ks_code == 1) return REHR_UNSUPPORTED;
  if (x.ld % 8 != 0) return REHR_BAD_ALIGNMENT;
  p.out = y.ptr;
  p.out_f32 = y_is_f32;
  p.out_f16 = y.dtype == REHR_F16;
  p.range = range_target(!y_is_f32 && p.out_f16);
  p.in_f16 = x.dtype == REHR_F16;
  p.out_ld = y.ld;
  p.o_pw = y.ld;
  p.o_ph = (long long)y.w * y.ld;
  p.o_pd = (long long)y.h * p.o_ph;
  p.o_pn = (long long)y.d * p.o_pd;
  if (ext) {
    const int R = (ks - 1) / 2;
    for (int a = 0; a < 3; ++a)
      if (ext->lo[a] > R || ext->hi[a] < R || ext->lo[a] < 0 || ext->hi[a] > ks - 1) return REHR_UNSUPPORTED;  // centre tap must exist
    p.kd_lo = ext->lo[0]; p.kd_hi = ext->hi[0];
    p.kh_lo = ext->lo[1]; p.kh_hi = ext->hi[1];
    p.kw_lo = ext->lo[2]; p.kw_hi = ext->hi[2];
    p.o_pn = ext->pn; p.o_pd = ext->pd; p.o_ph = ext->ph; p.o_pw = ext->pw;
    p.OD = ext->OD; p.OH = ext->OH; p.OW = ext->OW;
    if ((p.o_pw | p.o_ph | p.o_pd | p.o_pn) & 7) return REHR_BAD_ALIGNMENT;
  }
  p.bias = bias;
  p.act = act;
  p.slope = slope;
  p.stats = stats;
  p.err = nullptr;
  {
    const char* dbg = getenv("REHR_MARCH_DEBUG");
    p.debug = dbg ? atoi(dbg) : 0;
    static long long* prof_buf = nullptr;
    if (getenv("REHR_MARCH_PROF")) {
      if (!prof_buf) cudaMalloc(&prof_buf, 16 * sizeof(long long));
      long long h[16];
      if (cudaMemcpy(h, prof_buf, sizeof(h), cudaMemcpyDeviceToHost) == cudaSuccess && h[7] > 0 && h[7] < (1LL << 40))
        fprintf(stderr, "[march prof, previous launch, CTA0] producer wait_empty %.0f/plane (%lld) | mma wait_tempty %.0f wait_full %.0f issue+commit %.0f /plane (%lld) | epi wait_tfull %.0f body %.0f /plane (%lld)\n",
                (double)h[0] / h[1], h[1], (double)h[4] / h[7], (double)h[5] / h[7], (double)h[6] / h[7], h[7], (double)h[8] / h[10], (double)h[9] / h[10], h[10]);
      cudaMemset(prof_buf, 0, 16 * sizeof(long long));
      p.prof = prof_buf;
    }
  }
  {
    const unsigned long long gdim[5] = {(unsigned long long)x.c, (unsigned long long)x.w, (unsigned long long)x.h,
                                        (unsigned long long)x.d, (unsigned long long)x.n};
    const unsigned long long pitch = (unsigned long long)x.ld * 2;
    const unsigned long long gstr[4] = {pitch, pitch * x.w, pitch * x.w * x.h, pitch * x.w * x.h * x.d};
    const unsigned box[5] = {(unsigned)p.BK, (unsigned)(kTileW + ks - 1), (unsigned)(kTileH + ks - 1), 1u, 1u};
    rc = encode_tiled_bf16(&p.x_map, x.ptr, 5, gdim, gstr, box, p.BK * 2);
    if (rc != REHR_OK) return rc;
  }
  {
    const unsigned long long rows = (unsigned long long)p.n_ct * ks * ks * p.chunks * p.wrows;
    const unsigned long long gdim[2] = {(unsigned long long)p.BK, rows};
    const unsigned long long gstr[1] = {(unsigned long long)p.BK * 2};
    const unsigned box[2] = {(unsigned)p.BK, (unsigned)p.wrows};
    rc = encode_tiled_bf16(&p.w_map, w_march, 2, gdim, gstr, box, p.BK * 2);
    if (rc != REHR_OK) return rc;
  }
  return dispatch_march(pl, stream);
}

template <int BKT, int CHUNKS, int CT, int KS>
static int launch_variant(const MarchPlan& pl, cudaStream_t stream) {
  if (pl.p.range != nullptr) {
    REHR_SET_MAX_SMEM_ONCE((conv_march_kernel<BKT, CHUNKS, CT, KS, true>), 227 * 1024);
    conv_march_kernel<BKT, CHUNKS, CT, KS, true><<<pl.grid, kMarchThreads, pl.smem, stream>>>(pl.p);
  } else {
    REHR_SET_MAX_SMEM_ONCE((conv_march_kernel<BKT, CHUNKS, CT, KS, false>), 227 * 1024);
    conv_march_kernel<BKT, CHUNKS, CT, KS, false><<<pl.grid, kMarchThreads, pl.smem, stream>>>(pl.p);
  }
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

static int dispatch_march(const MarchPlan& pl, cudaStream_t stream) {
  const int bk = pl.p.BK, ch = pl.p.chunks, ct = pl.p.Ct, ks = pl.p.ks;
  if (ks == 5) {
    if (bk == 16 && ch == 1 && ct == 16) return launch_variant<16, 1, 16, 5>(pl, stream);
    return REHR_UNSUPPORTED;
  }
#define REHR_MARCH_CASE(B, C, T) \
  if (bk == B && ch == C && ct == T) return launch_variant<B, C, T, 3>(pl, stream);
  REHR_MARCH_CASE(16, 1, 16)
  REHR_MARCH_CASE(16, 1, 32)
  REHR_MARCH_CASE(16, 1, 64)
  REHR_MARCH_CASE(32, 1, 16)
  REHR_MARCH_CASE(32, 1, 32)
  REHR_MARCH_CASE(32, 1, 64)
  REHR_MARCH_CASE(64, 1, 16)
  REHR_MARCH_CASE(64, 1, 32)
  REHR_MARCH_CASE(64, 2, 16)
  REHR_MARCH_CASE(64, 1, 64)  // planar 64 -> 64
  REHR_MARCH_CASE(64, 2, 32)  // planar 128 -> 64
#undef REHR_MARCH_CASE
  return REHR_UNSUPPORTED;
}

// ------------------------------------------------------------------------------------------------
// Weight packing for the marching kernel (T = KS^3 taps):
//   dst[ct][khw][chunk][j*Ct + col][BK]   with  j = KS-1 - kd,  co = ct*Ct + col (zero rows for co >= cout),  ci = chunk*BK + k
//   src element = w[co*s_co + ci*s_ci + (flip ? T-1 - t : t)],  t = (kd*KS + kh)*KS + kw
// forward of W[Cout][Cin][T]: s_co = Cin*T, s_ci = T, flip = 0;
// input-gradient (dx[B] from dy[A]) of W[A][B][T]: cout := B, cin := A, s_co = T, s_ci = B*T, flip = 1.
// ------------------------------------------------------------------------------------------------
__global__ void pack_march_kernel(const float* __restrict__ src, unsigned short* __restrict__ dst, int cout, int cout_pad, int cin,
                                  int Ct, int BK, int ks, int kdn, long long s_co, long long s_ci, int flip, int f16) {
  // kdn = stored depth taps: ks (cubic kernel) or 1 (planar k(1,ks,ks): source taps t = kh*ks + kw)
  const int chunks = cin / BK;
  const int T = kdn * ks * ks;
  const long long total = (long long)cout_pad * cin * T;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i % BK);
    long long r = i / BK;
    const int rowi = (int)(r % (kdn * Ct));
    r /= kdn * Ct;
    const int chunk = (int)(r % chunks);
    r /= chunks;
    const int khw = (int)(r % (ks * ks));
    const int ct = (int)(r / (ks * ks));
    const int j = rowi / Ct, col = rowi % Ct;
    const int kd = kdn - 1 - j, kh = khw / ks, kw = khw % ks;
    const int t = (kd * ks + kh) * ks + kw;
    const int co = ct * Ct + col, ci = chunk * BK + k;
    dst[i] = co < cout ? pack16(src[co * s_co + ci * s_ci + (flip ? T - 1 - t : t)], f16) : (unsigned short)0;
  }
}

// Packed weights of the 8 (or 4 / 2) output parity classes of the input gradient of a k3 / pad 1 conv with strides in {1, 2}:
// class r of a stride-2 dimension sees a stride-1 correlation over dy with tap u (offset u - 1): r = 0 -> {u=1: k=1};
// r = 1 -> {u=1: k=2, u=2: k=0}; a stride-1 dimension has the ordinary flipped taps u -> k = 2 - u.  Taps a class does not
// use are zero (and skipped by the kernel through its tap ranges).  src = conv weight W[A][B][27] (A = conv Cout = channels
// of dy, B = conv Cin = channels of dx); marching "cin" = A, "cout" = B.  dst = [class][ct][khw][chunk][j*Ct + col][BK].
__global__ void pack_march_s2dgrad_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int A, int B, int Bpad,
                                          int Ct, int BK, int sd, int sh, int sw) {
  const int chunks = A / BK;
  const long long per_cls = (long long)Bpad * A * 27;
  const int ncls = sd * sh * sw;
  const long long total = per_cls * ncls;
  for (long long i0 = blockIdx.x * (long long)blockDim.x + threadIdx.x; i0 < total; i0 += (long long)gridDim.x * blockDim.x) {
    const int cls = (int)(i0 / per_cls);
    long long i = i0 % per_cls;
    const int rw = cls % sw, rh = (cls / sw) % sh, rd = cls / (sw * sh);
    const int k = (int)(i % BK);
    long long r = i / BK;
    const int rowi = (int)(r % (3 * Ct));
    r /= 3 * Ct;
    const int chunk = (int)(r % chunks);
    r /= chunks;
    const int khw = (int)(r % 9);
    const int ct = (int)(r / 9);
    const int j = rowi / Ct, col = rowi % Ct;
    const int u[3] = {2 - j, khw / 3, khw % 3};
    const int st[3] = {sd, sh, sw}, rr[3] = {rd, rh, rw};
    int kk[3];
    bool ok = true;
    for (int a = 0; a < 3; ++a) {
      if (st[a] == 1) kk[a] = 2 - u[a];
      else if (rr[a] == 0) { kk[a] = 1; ok = ok && u[a] == 1; }
      else { kk[a] = u[a] == 1 ? 2 : 0; ok = ok && u[a] >= 1; }
    }
    const int b = ct * Ct + col, a_ch = chunk * BK + k;
    float v = 0.f;
    if (ok && b < B) v = src[((long long)a_ch * B + b) * 27 + (kk[0] * 3 + kk[1]) * 3 + kk[2]];
    dst[i0] = __float2bfloat16(v);
  }
}

}  // namespace rehr

using namespace rehr;

// 3 / 5: cubic kernel; 1: planar k(1,3,3) pad (0,1,1); 0: not a marching layer
static int march_ks_of(const rehr_conv_desc* d) {
  if (!d) return 0;
  if (d->kd == 1 && d->kh == 3 && d->kw == 3 && d->sd == 1 && d->sh == 1 && d->sw == 1 && d->pd == 0 && d->ph == 1 && d->pw == 1) return 1;
  if (d->kd != d->kh || d->kh != d->kw || (d->kd != 3 && d->kd != 5)) return 0;
  if (d->sd != 1 || d->sh != 1 || d->sw != 1) return 0;
  const int r = (d->kd - 1) / 2;
  if (d->pd != r || d->ph != r || d->pw != r) return 0;
  return d->kd;
}

extern "C" {

int rehr_conv3d_march_supported(const rehr_conv_desc* d, int cin, int cout) {
  const int ks = march_ks_of(d);
  if (ks == 0) return 0;
  return march_ct(cin, cout, ks == 1 ? 3 : ks, ks == 1) > 0 ? 1 : 0;
}

// ks: 3 / 5 = cubic kernel, 1 = planar k(1,3,3) (the kernel's depth extent, as in the other marching entry points)
size_t rehr_conv3d_march_weight_bytes(int cin, int cout, int ks) {
  if (ks == 1) return march_ct(cin, cout, 3, true) > 0 ? (size_t)9 * cin * pad16(cout) * 2 : 0;
  return march_ct(cin, cout, ks, false) > 0 ? (size_t)ks * ks * ks * cin * pad16(cout) * 2 : 0;
}

int rehr_pack_weight_march(const float* src, void* dst16, int cout, int cin, int ks, long long s_co, long long s_ci, int flip,
                           int dtype, rehr_stream stream) {
  if (!src || !dst16) return REHR_BAD_SHAPE;
  const bool planar = ks == 1;
  if (planar) ks = 3;
  const int kdn = planar ? 1 : ks;
  const int ct = march_ct(cin, cout, ks, planar);
  if (ct == 0) return REHR_UNSUPPORTED;
  const long long total = (long long)pad16(cout) * cin * kdn * ks * ks;
  if (pack_recording()) {
    PackJob j{};
    j.src = src; j.dst = dst16; j.kind = 1; j.f16 = dtype == REHR_F16; j.total = total;
    j.cout = cout; j.cout_pad = pad16(cout); j.cin = cin; j.Ct = ct; j.BK = std::min(cin, 64); j.ks = ks; j.kdn = kdn;
    j.s_co = s_co; j.s_ci = s_ci; j.flip = flip;
    return pack_record(j);
  }
  const int blocks = (int)std::min<long long>((total + 255) / 256, 148 * 16);
  pack_march_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(src, reinterpret_cast<unsigned short*>(dst16), cout, pad16(cout), cin, ct,
                                                             std::min(cin, 64), ks, kdn, s_co, s_ci, flip, dtype == REHR_F16);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_conv3d_march_stats_tiles(const rehr_tensor* x, const rehr_tensor* y, int ks) {
  if (!x || !y) return 0;
  return march_stats_tiles(*x, *y, ks);
}

int rehr_conv3d_march_fwd(const rehr_tensor* x, const void* w_march, const float* bias, const rehr_tensor* y, int ks, int y_is_f32,
                          int act, float slope, float* stats, rehr_stream stream) {
  if (!x || !y || !x->ptr || !y->ptr || !w_march) return REHR_BAD_SHAPE;
  return launch_march(*x, w_march, bias, *y, ks, y_is_f32, act, slope, stats, (cudaStream_t)stream);
}

// ---- stride-2 (per dimension 1 or 2) input gradient of a k3 / pad 1 conv through the marching kernel, one launch per parity class
static bool s2dgrad_desc_ok(const rehr_conv_desc* d) {
  if (!d) return false;
  if (d->kd != 3 || d->kh != 3 || d->kw != 3 || d->pd != 1 || d->ph != 1 || d->pw != 1) return false;
  if ((d->sd != 1 && d->sd != 2) || (d->sh != 1 && d->sh != 2) || (d->sw != 1 && d->sw != 2)) return false;
  return d->sd * d->sh * d->sw > 1;
}
int rehr_conv3d_march_s2dgrad_supported(const rehr_conv_desc* d, int cin, int cout) {
  return s2dgrad_desc_ok(d) && march_ct(cout, cin, 3, false) > 0 ? 1 : 0;  // marching cin = conv Cout (dy), cout = conv Cin (dx)
}
size_t rehr_conv3d_march_s2dgrad_weight_bytes(const rehr_conv_desc* d, int cin, int cout) {
  if (!rehr_conv3d_march_s2dgrad_supported(d, cin, cout)) return 0;
  return (size_t)d->sd * d->sh * d->sw * 27 * cout * pad16(cin) * 2;
}
int rehr_pack_weight_march_s2dgrad(const rehr_conv_desc* d, const float* w, void* dst_bf16, int cin, int cout, rehr_stream stream) {
  if (!w || !dst_bf16) return REHR_BAD_SHAPE;
  if (!rehr_conv3d_march_s2dgrad_supported(d, cin, cout)) return REHR_UNSUPPORTED;
  const int ct = march_ct(cout, cin, 3, false);
  const long long total = (long long)d->sd * d->sh * d->sw * 27 * cout * pad16(cin);
  if (pack_recording()) {
    PackJob j{};
    j.src = w; j.dst = dst_bf16; j.kind = 2; j.f16 = 0; j.total = total;
    j.cin = cout; j.cout = cin; j.cout_pad = pad16(cin); j.Ct = ct; j.BK = std::min(cout, 64);   // A = conv Cout, B = conv Cin
    j.sd = d->sd; j.sh = d->sh; j.sw = d->sw;
    return pack_record(j);
  }
  const int blocks = (int)std::min<long long>((total + 255) / 256, 148 * 16);
  pack_march_s2dgrad_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(w, reinterpret_cast<__nv_bfloat16*>(dst_bf16), cout, cin, pad16(cin),
                                                                      ct, std::min(cout, 64), d->sd, d->sh, d->sw);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}
int rehr_conv3d_march_s2dgrad(const rehr_conv_desc* d, const rehr_tensor* dy, const void* w_packed, const rehr_tensor* dx,
                              rehr_stream stream) {
  if (!dy || !dx || !dy->ptr || !dx->ptr || !w_packed) return REHR_BAD_SHAPE;
  if (!rehr_conv3d_march_s2dgrad_supported(d, dx->c, dy->c)) return REHR_UNSUPPORTED;
  const int s[3] = {d->sd, d->sh, d->sw};
  const int in[3] = {dx->d, dx->h, dx->w}, out[3] = {dy->d, dy->h, dy->w};
  for (int a = 0; a < 3; ++a)
    if (out[a] != (in[a] + 2 - 3) / s[a] + 1) return REHR_BAD_SHAPE;
  if (dx->n != dy->n || dx->ld % 8 != 0) return REHR_BAD_SHAPE;
  const size_t per_cls = (size_t)27 * dy->c * pad16(dx->c) * 2;
  const long long pw = dx->ld, ph = (long long)dx->w * pw, pd = (long long)dx->h * ph, pn = (long long)dx->d * pd;
  int cls = 0;
  for (int rd = 0; rd < s[0]; ++rd)
    for (int rh = 0; rh < s[1]; ++rh)
      for (int rw = 0; rw < s[2]; ++rw, ++cls) {
        const int r[3] = {rd, rh, rw};
        MarchExt e;
        int ext[3];
        bool empty = false;
        for (int a = 0; a < 3; ++a) {
          ext[a] = (in[a] - r[a] + s[a] - 1) / s[a];
          if (ext[a] <= 0) empty = true;
          if (s[a] == 1) { e.lo[a] = 0; e.hi[a] = 2; }
          else if (r[a] == 0) { e.lo[a] = 1; e.hi[a] = 1; }
          else { e.lo[a] = 1; e.hi[a] = 2; }
        }
        if (empty) continue;
        e.pn = pn; e.pd = pd * s[0]; e.ph = ph * s[1]; e.pw = pw * s[2];
        e.OD = ext[0]; e.OH = ext[1]; e.OW = ext[2];
        // the class is computed on the dy grid; its rows are written at (2i + r) of dx
        rehr_tensor yv = *dy;  // output "tensor" of the marching conv: dy grid, dx channels, class base pointer
        yv.c = dx->c;
        yv.ld = dx->ld;
        yv.ptr = reinterpret_cast<__nv_bfloat16*>(dx->ptr) + rd * pd + rh * ph + rw * pw;
        int rc = launch_march(*dy, reinterpret_cast<const uint8_t*>(w_packed) + cls * per_cls, nullptr, yv, 3, 0, REHR_ACT_NONE, 0.f,
                              nullptr, (cudaStream_t)stream, &e);
        if (rc != REHR_OK) return rc;
      }
  return REHR_OK;
}

}  // extern "C"
