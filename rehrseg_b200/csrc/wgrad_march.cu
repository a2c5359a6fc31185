// "Marching" weight-gradient kernel for sm_100a: k = 3x3x3, stride 1, pad 1 layers (the ones that hold 3/4 of the
// nnU-Net FLOPs -- SURVEY.md section 7.3).  Companion of conv_march.cu (forward / input-gradient).
//
//   dW[co][ci][kd][kh][kw] = sum_{n,d,h,w} dY[n,d,h,w,co] * X[n,d+kd-1,h+kh-1,w+kw-1,ci]
//
// is a GEMM whose K dimension is the VOXEL index, so both operands are "MN-major" views of the channels-last
// activation tiles exactly as TMA writes them (no transposes, no im2col).  Of the two tensors one plays the halo
// operand Hh (M side) and the other the plain operand Pp (N side); per CTA and per input plane q the kernel computes
//
//   G[a][j][ch][cp] += sum_{u in 16x8 tile} Hh[q][u + off(a) - (1,1)][ch] * Pp[q-1+j][u][cp],   a = 3*oh+ow in 0..8, j in 0..2
//
//   * Hh plane q is TMA-loaded ONCE as an 18x10 halo'd tile (CH = 32 or 64 channels of it); the 9 in-plane offsets are
//     NOT re-loaded: they are row shifts folded into the UMMA descriptor start address, and 128/CH of them are stacked
//     along M through the descriptor's leading-dimension byte offset (LBO = the row distance between two offsets) --
//     verified on B200 by tools/umma_probe_mn.cu (profiles/r01_umma_mn_major_probe.log);
//   * the three depth offsets are fused along N: Pp planes q-1, q, q+1 (32 channels each) sit in adjacent slots of a
//     shared-memory ring (slots 0,1 are mirrored behind the last slot so the triple is always contiguous), one
//     tcgen05.mma has N = 96;
//   * the accumulators (groups x 96 columns x 128 lanes fp32) stay in TMEM for the whole life of the CTA: there is
//     no epilogue inside the loop, the MMA thread issues back to back, and each CTA writes one partial dW at the end;
//     a second tiny kernel sums the <= 148 partials (deterministic order, no atomics) and scatters into PyTorch layout.
// Role A: Hh = X, Pp = dY  (kh = oh, kw = ow, kd = 2-j);   role B: Hh = dY, Pp = X  (kh = 2-oh, kw = 2-ow, kd = j).
// Channel counts beyond one piece (CH of Hh, 32 of Pp) are covered by independent (h-split, p-split) "combos", each
// owned by its own set of CTAs.
//
// Reference call sites replaced: the weight-gradient half of torch.nn.Conv3d.backward for ConvDropoutNormReLU.conv of
// the full / half resolution stages (built at models/seg_model.py:174-191, driven by loss.backward() at
// train_all.py:555).
#include "engine.h"
#include "ptx.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace rehr {

int encode_tiled_bf16(CUtensorMap* m, const void* base, int rank, const unsigned long long* gdim,
                      const unsigned long long* gstride_bytes, const unsigned* box, int swizzle_bytes);

static constexpr int kWgmThreads = 192;  // warp0 TMA, warp1 MMA (+TMEM alloc), warps 2..5 TMEM zero / final drain
static constexpr int kWTileH = 16, kWTileW = 8;
// Plain-plane ring: KS planes are read by a step, the rest is prefetch distance.  Measured (profiles/r02_s2wgrad_ncu_summary.txt):
// neither 9 spare slots nor a 12-deep halo ring changes the stride-2 32->64 @128^3 weight gradient (0.64 ms either way): that
// launch is bound by the RATE at which TMA fetches the 64-byte granules of the parity-class views (13 B/clk/SM), not by latency.
static constexpr int kPSpare = 3;
static constexpr int kMaxHStages = 12;    // halo-plane ring: as deep as shared memory allows (WgmParams::h_stages, >= 4): the loop is
                                          // bound by TMA latency when a step issues few MMAs (parity classes of a stride-2 conv)

struct alignas(64) WgmParams {
  CUtensorMap h_map;  // 5-D NDHWC, box (CH, 8 + KS - 1, 16 + KS - 1, 1, 1)
  CUtensorMap p_map;  // 5-D NDHWC, box (PC, 8, 16, 1, 1)
  int N, D, H, W;
  int tiles_h, tiles_w, Ds, n_seg;
  int n_hs, n_ps, n_combo, ctas_per_combo, items_per_combo;
  uint32_t h_stride;  // bytes per halo stage (1024-aligned)
  int h_stages;       // halo ring depth
  // sub-setting for the parity classes of a stride-2 conv (rehr_conv3d_wgrad_march_s2): which MMA groups (in-plane offset rows)
  // and which of the fused depth planes j are needed; everything else would multiply zeros
  int g_mask, j_min, j_max;
  float* ws;          // [cta][group][128][KS * PC]
  int* err;
  // fused parity classes (n_cls > 0): CTAs [cls_begin[c], cls_begin[c + 1]) work on class c -- halo operand h_maps[c], its own
  // group mask / depth-plane range -- all inside ONE launch, so the TMEM drain and the partial-dW reduction are paid once per CTA
  // instead of once per class pass, and the 8 classes share the dY tiles through L2
  int n_cls;
  int cls_begin[9];
  int cls_gmask[8], cls_jmin[8], cls_jmax[8];
  CUtensorMap h_maps[8];
};

// Geometry of one (CH halo channels, PC plain channels, KS kernel size) variant.
//   * plain planes: KS consecutive ones (q - R .. q + R) are fused along N (= KS * PC); ring of KS + 3 slots with the
//     first KS - 1 mirrored behind the last one so that the KS-tuple is always contiguous in shared memory;
//   * halo tile: the KS in-plane offsets of one kernel row (kh) are consecutive tile rows, so they are stacked along M through
//     LBO = one row; 128 / CH of them fit one MMA ("part"); for CH = 64, KS = 3 the 9 offsets are paired freely instead
//     (any two rows form an arithmetic progression), which needs 5 MMAs instead of 6.
// JP = number of fused depth planes that own accumulator columns (default KS).  The parity classes of a stride-2 conv never use
// the plane q - 1 (j = 0), so JP = 2 there: N <= 2 * PC, which lets ONE piece cover all 64 dY channels (PC = 64, 3 x 128 TMEM
// columns) -- X is then streamed once instead of once per 32-channel dY piece, in 128-byte instead of 64-byte dY rows.
template <int CH, int PC, int KS, int JP = KS>
struct WgmCfg {
  static constexpr int R = (KS - 1) / 2;
  static constexpr int kHaloH = kWTileH + KS - 1, kHaloW = kWTileW + KS - 1, kHaloRows = kHaloH * kHaloW;
  static constexpr int kApm = 128 / CH;                   // atoms (in-plane offsets) per MMA
  static constexpr int kParts = (KS + kApm - 1) / kApm;   // MMAs per kernel row
  static constexpr bool kPaired = (CH == 64 && KS == 3);
  static constexpr int kGroups = kPaired ? 5 : KS * kParts;
  static constexpr int kN = JP * PC;                      // accumulator columns per group
  static constexpr int kJ0 = KS - JP;                     // first fused plane index that owns accumulator columns
  static constexpr uint32_t kRowB = CH * 2;
  static constexpr uint32_t kLayout = kRowB == 128 ? 2u : (kRowB == 64 ? 4u : 6u);
  static constexpr uint32_t kPRowB = PC * 2;
  static constexpr uint32_t kPLayout = kPRowB == 128 ? 2u : (kPRowB == 64 ? 4u : 6u);
  static constexpr uint32_t kPSlotBytes = kWTileH * kWTileW * PC * 2;
  static constexpr int kPRing = KS + kPSpare, kMirror = KS - 1;
  static_assert(kGroups * kN <= 512, "accumulators must fit TMEM");
  __host__ __device__ static constexpr int row0(int g) {
    return kPaired ? ((2 * g) / 3) * kHaloW + (2 * g) % 3 : (g / kParts) * kHaloW + (g % kParts) * kApm;
  }
  __host__ __device__ static constexpr int lbo_rows(int g) {
    if (!kPaired || g == 4) return 1;
    const int a0 = 2 * g, a1 = 2 * g + 1;
    return ((a1 / 3) * kHaloW + a1 % 3) - ((a0 / 3) * kHaloW + a0 % 3);
  }
};

__device__ __forceinline__ bool wgm_elect() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}

struct WgmItem {
  int n, seg, th, tw;
};
__device__ __forceinline__ WgmItem wgm_decode(const WgmParams& p, int item) {
  WgmItem c;
  c.tw = item % p.tiles_w;
  item /= p.tiles_w;
  c.th = item % p.tiles_h;
  item /= p.tiles_h;
  c.seg = item % p.n_seg;
  c.n = item / p.n_seg;
  return c;
}

template <int CH, int PC, int KS, int JP = KS>
__global__ void __launch_bounds__(kWgmThreads, 1) wgrad_march_kernel(const __grid_constant__ WgmParams p) {
  using Cfg = WgmCfg<CH, PC, KS, JP>;
  constexpr int R = Cfg::R;
  constexpr int kPRing = Cfg::kPRing;
  constexpr uint32_t kPSlotBytes = Cfg::kPSlotBytes;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* s_p = smem;                                                    // (kPRing + kMirror) plain-plane slots
  uint8_t* s_h = smem + (((size_t)(kPRing + Cfg::kMirror) * kPSlotBytes + 1023) & ~size_t(1023));  // kHStages x h_stride
  const uint32_t kHStages = (uint32_t)p.h_stages;
  uint8_t* tail = s_h + (size_t)kHStages * p.h_stride;
  uint64_t* full_h = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_h = full_h + kMaxHStages;
  uint64_t* full_p = empty_h + kMaxHStages;
  uint64_t* empty_p = full_p + kPRing;
  uint64_t* zero_bar = empty_p + kPRing;
  uint64_t* done_bar = zero_bar + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    if (p.n_cls == 0) tma_prefetch_desc(&p.h_map);
    tma_prefetch_desc(&p.p_map);
    for (int i = 0; i < kMaxHStages; ++i) {
      mbar_init(&full_h[i], 1);
      mbar_init(&empty_h[i], 1);
    }
    for (int i = 0; i < kPRing; ++i) {
      mbar_init(&full_p[i], 1);
      mbar_init(&empty_p[i], 1);
    }
    mbar_init(zero_bar, 4);
    mbar_init(done_bar, 1);
    fence_mbar_init();
  } else if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // class (fused stride-2 passes) -> CTA range, halo map, masks; a single class otherwise
  int cta = blockIdx.x, ctas_per_combo = p.ctas_per_combo;
  int g_mask = p.g_mask, j_min = p.j_min, j_max = p.j_max;
  const CUtensorMap* h_map = &p.h_map;
  int cls = 0;
  if (p.n_cls > 0) {
    while (cls + 1 < p.n_cls && (int)blockIdx.x >= p.cls_begin[cls + 1]) ++cls;
    cta = blockIdx.x - p.cls_begin[cls];
    ctas_per_combo = (p.cls_begin[cls + 1] - p.cls_begin[cls]) / p.n_combo;
    g_mask = p.cls_gmask[cls];
    j_min = p.cls_jmin[cls];
    j_max = p.cls_jmax[cls];
    h_map = &p.h_maps[cls];
  }
  const int combo = cta % p.n_combo;
  const int rank = cta / p.n_combo;
  const int hs = combo / p.n_ps, ps = combo % p.n_ps;

  if (warp == 0) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      uint32_t kh = 0, kp = 0;  // running plane counters (ring position = counter % ring, parity = (counter / ring) & 1)
      for (int item = rank; item < p.items_per_combo; item += ctas_per_combo) {
        const WgmItem c = wgm_decode(p, item);
        const int d0 = c.seg * p.Ds, d1 = min(p.D, d0 + p.Ds);
        const int pa = max(d0 - R, 0), pb = min(d1 - 1 + R, p.D - 1);
        const int h0 = c.th * kWTileH, w0 = c.tw * kWTileW;
        int next_p = pa;
        for (int q = d0; q < d1; ++q) {
          const int need = min(q + R, pb);
          while (next_p <= need) {
            const uint32_t slot = kp % kPRing;
            const bool mirrored = slot < (uint32_t)Cfg::kMirror;
            mbar_wait(&empty_p[slot], ((kp / kPRing) & 1u) ^ 1u, p.err, 51);
            mbar_arrive_expect_tx(&full_p[slot], mirrored ? 2 * kPSlotBytes : kPSlotBytes);
            tma_load_5d(&p.p_map, &full_p[slot], s_p + (size_t)slot * kPSlotBytes, ps * PC, w0, h0, next_p, c.n);
            if (mirrored)
              tma_load_5d(&p.p_map, &full_p[slot], s_p + (size_t)(slot + kPRing) * kPSlotBytes, ps * PC, w0, h0, next_p, c.n);
            ++kp;
            ++next_p;
          }
          const uint32_t st = kh % kHStages;
          mbar_wait(&empty_h[st], ((kh / kHStages) & 1u) ^ 1u, p.err, 52);
          mbar_arrive_expect_tx(&full_h[st], Cfg::kHaloRows * Cfg::kRowB);
          tma_load_5d(h_map, &full_h[st], s_h + (size_t)st * p.h_stride, hs * CH, w0 - R, h0 - R, q, c.n);
          ++kh;
        }
      }
    }
  } else if (warp == 1) {
    // ============================== MMA issuer ==============================
    // descriptor high words: SBO (bits 32..45) = pitch between 8-voxel groups, version 1 (bit 46), swizzle (61..63)
    constexpr uint32_t kAHi = ((Cfg::kHaloW * Cfg::kRowB) >> 4) | (1u << 14) | (Cfg::kLayout << 29);
    constexpr uint32_t kBHi = ((8u * Cfg::kPRowB) >> 4) | (1u << 14) | (Cfg::kPLayout << 29);
    constexpr uint32_t kBLoLbo = (kPSlotBytes >> 4) << 16;
    const uint32_t sp_lo = smem_u32(s_p) >> 4, sh_lo = smem_u32(s_h) >> 4;
    const uint32_t hstride_lo = p.h_stride >> 4;
    mbar_wait(zero_bar, 0, p.err, 61);  // accumulators zeroed by the drain warps
    tc_fence_after();
    uint32_t kh = 0, kp = 0;
    for (int item = rank; item < p.items_per_combo; item += ctas_per_combo) {
      const WgmItem c = wgm_decode(p, item);
      const int d0 = c.seg * p.Ds, d1 = min(p.D, d0 + p.Ds);
      const int pa = max(d0 - R, 0), pb = min(d1 - 1 + R, p.D - 1);
      const uint32_t cnt0 = kp;  // counter of plane pa
      int waited = pa - 1;
      for (int q = d0; q < d1; ++q) {
        const int need = min(q + R, pb);
        while (waited < need) {
          ++waited;
          const uint32_t cc = cnt0 + (uint32_t)(waited - pa);
          mbar_wait(&full_p[cc % kPRing], (cc / kPRing) & 1u, p.err, 62);
        }
        const uint32_t st = kh % kHStages;
        mbar_wait(&full_h[st], (kh / kHStages) & 1u, p.err, 63);
        tc_fence_after();
        // plain planes q - R + j, j in [jlo, jhi], exist inside the volume
        const int jlo = max(max(0, R - q), j_min), jhi = min(min(KS - 1, p.D - 1 - q + R), j_max);
        const uint32_t cbase = cnt0 + (uint32_t)(q - R + jlo - pa);
        const uint32_t s0 = cbase % kPRing;
        const uint32_t idesc = make_idesc_bf16(128, max(jhi - jlo + 1, 1) * PC, 1, 1);
        const uint32_t a_lo = sh_lo + st * hstride_lo;
        const uint32_t b_lo = (sp_lo + s0 * (kPSlotBytes >> 4)) | kBLoLbo;
        const uint32_t d_tmem = tmem_base + (uint32_t)((jlo - Cfg::kJ0) * PC);   // host guarantees j_min >= kJ0
        if (wgm_elect()) {
          if (jlo <= jhi) {
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) {
              const uint64_t bd = ((uint64_t)kBHi << 32) | (uint64_t)(b_lo + (uint32_t)((ks * 16 * Cfg::kPRowB) >> 4));
#pragma unroll
              for (int g = 0; g < Cfg::kGroups; ++g) {
                if (!((g_mask >> g) & 1)) continue;
                const uint32_t a_off = (uint32_t)(((2 * ks * Cfg::kHaloW + Cfg::row0(g)) * Cfg::kRowB) >> 4) |
                                       ((uint32_t)((Cfg::lbo_rows(g) * Cfg::kRowB) >> 4) << 16);
                const uint64_t ad = ((uint64_t)kAHi << 32) | (uint64_t)(a_lo + a_off);
                umma_bf16(d_tmem + (uint32_t)(g * Cfg::kN), ad, bd, idesc, 1u);
              }
            }
          }
          umma_commit(&empty_h[st]);
          // plain planes whose last reader is this step
          if (q - R >= pa) umma_commit(&empty_p[(cnt0 + (uint32_t)(q - R - pa)) % kPRing]);
          if (q == d1 - 1) {
            for (int r = max(q - R + 1, pa); r <= pb; ++r) umma_commit(&empty_p[(cnt0 + (uint32_t)(r - pa)) % kPRing]);
          }
        }
        __syncwarp();
        ++kh;
      }
      kp = cnt0 + (uint32_t)(pb - pa + 1);
    }
    if (wgm_elect()) umma_commit(done_bar);
    __syncwarp();
  } else {
    // ============================== TMEM zero, then final drain (warps 2..5) ==============================
    const int q4 = warp & 3;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q4 * 32) << 16);
    {
      uint32_t z[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) z[i] = 0u;
      for (int c0 = 0; c0 < 512; c0 += 32) tmem_st32(lane_addr + (uint32_t)c0, z);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(zero_bar);
    }
    mbar_wait(done_bar, 0, p.err, 71);
    tc_fence_after();
    const int row = q4 * 32 + lane;
    float* dst = p.ws + ((size_t)blockIdx.x * Cfg::kGroups * 128 + row) * Cfg::kN;
    for (int g = 0; g < Cfg::kGroups; ++g) {
#pragma unroll
      for (int c0 = 0; c0 < Cfg::kN; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(lane_addr + (uint32_t)(g * Cfg::kN + c0), v);
        tmem_ld_wait();
        float4* o = reinterpret_cast<float4*>(dst + (size_t)g * 128 * Cfg::kN + c0);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          o[i] = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]), __uint_as_float(v[4 * i + 2]),
                             __uint_as_float(v[4 * i + 3]));
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
// partial sums -> dW (PyTorch layout [co][ci][KS^3], fp32)
// ------------------------------------------------------------------------------------------------
struct WgmReduceParams {
  const float* ws;
  float* dw;
  int CH, PC, KS, JP, groups, apm, parts, paired;
  int n_hs, n_ps, n_combo, ctas_per_combo;
  int role;  // 0: Hh = X (ch = ci, cp = co), 1: Hh = dY (ch = co, cp = ci)
  int Ci, Co;        // channels of the dW tensor (Co may be smaller than the padded dY the kernel saw)
  int accumulate;
  // stride-2 parity class (rehr_conv3d_wgrad_march_s2): per dim (d h w) stride s and class r; offset e = k_stride1 - 1 maps
  // to the conv tap 2e + r + 1 (s = 2) or e + 1 (s = 1); offsets that give no tap in [0, 3) are dropped
  int cls_s[3], cls_r[3];
  // planar k(1,3,3) layer: only the centre depth offset was accumulated (j_min = j_max = 1); dW is [co][ci][9]
  int planar;
};

// Two thread layouts over the same index space (hs, ps, a, j, ch, cpl):
//   SLICED = true : block = PC (cpl) x 256/PC slices of a LONG partial list (one (.., ch) per block, shared-memory combine);
//   SLICED = false: block = PC (cpl) x 256/PC consecutive ch, every thread walks its SHORT partial list alone.
template <bool SLICED>
__global__ void __launch_bounds__(256) wgrad_march_reduce_kernel(const WgmReduceParams p) {
  __shared__ float red[16][65];   // [256 / PC slices][PC plain channels]: PC <= 64
  const int cpl = threadIdx.x % p.PC, sub = threadIdx.x / p.PC;
  const int nsub = 256 / p.PC;
  int idx = blockIdx.x;
  int ch;
  if (SLICED) {
    ch = idx % p.CH;
    idx /= p.CH;
  } else {
    const int chb = (p.CH + nsub - 1) / nsub;  // channel blocks per (.., j)
    ch = (idx % chb) * nsub + sub;
    idx /= chb;
  }
  const int j = idx % p.KS;
  idx /= p.KS;
  const int a = idx % (p.KS * p.KS);
  idx /= p.KS * p.KS;
  const int ps = idx % p.n_ps;
  const int hs = idx / p.n_ps;
  const int oh = a / p.KS, ow = a % p.KS;
  int g, at;
  if (p.paired) {
    g = a / 2;
    at = a % 2;
  } else {
    g = oh * p.parts + ow / p.apm;
    at = ow % p.apm;
  }
  const bool chok = ch < p.CH;
  const int m = at * p.CH + (chok ? ch : 0);
  const int kn = p.JP * p.PC;
  const int jc = j - (p.KS - p.JP);      // accumulator column block of fused plane j (planes below KS - JP own none)
  if (jc < 0) return;
  const int combo = hs * p.n_ps + ps;
  const size_t per_cta = (size_t)p.groups * 128 * kn;
  const size_t off = ((size_t)g * 128 + m) * kn + jc * p.PC + cpl;
  float t = 0.f;
  if (SLICED) {
    float acc = 0.f;
    for (int k = sub; k < p.ctas_per_combo; k += nsub) acc += p.ws[(size_t)(k * p.n_combo + combo) * per_cta + off];
    red[sub][cpl] = acc;
    __syncthreads();
    if (sub != 0) return;
    for (int s = 0; s < nsub; ++s) t += red[s][cpl];
  } else {
    if (!chok) return;
    for (int k = 0; k < p.ctas_per_combo; ++k) t += p.ws[(size_t)(k * p.n_combo + combo) * per_cta + off];
  }
  const int chH = hs * p.CH + ch, chP = ps * p.PC + cpl;
  int co, ci, kd, kh, kw;
  if (p.role == 0) {
    ci = chH; co = chP; kh = oh; kw = ow; kd = p.KS - 1 - j;
  } else {
    co = chH; ci = chP; kh = p.KS - 1 - oh; kw = p.KS - 1 - ow; kd = j;
  }
  if (p.cls_s[0] > 0) {
    int kk[3] = {kd, kh, kw};
    for (int a3 = 0; a3 < 3; ++a3) {
      const int e = kk[a3] - 1;
      const int t = p.cls_s[a3] == 2 ? 2 * e + p.cls_r[a3] + 1 : e + 1;
      if (t < 0 || t > 2) return;
      kk[a3] = t;
    }
    kd = kk[0]; kh = kk[1]; kw = kk[2];
  }
  if (p.planar) {
    if (kd != 1) return;
    if (co < p.Co && ci < p.Ci) {
      float* d = p.dw + ((size_t)co * p.Ci + ci) * 9 + kh * 3 + kw;
      *d = p.accumulate ? (*d + t) : t;
    }
    return;
  }
  if (co < p.Co && ci < p.Ci) {
    float* d = p.dw + ((size_t)co * p.Ci + ci) * (p.KS * p.KS * p.KS) + (kd * p.KS + kh) * p.KS + kw;
    *d = p.accumulate ? (*d + t) : t;
  }
}

// ------------------------------------------------------------------------------------------------
// host planning
// ------------------------------------------------------------------------------------------------
struct WgmPlan {
  WgmParams p;
  int CH, PC, KS, JP, role, grid, groups, planar;
  size_t smem, ws_bytes;
};

static int wgm_groups(int ch, int ks) {
  if (ch == 64 && ks == 3) return 5;
  const int apm = 128 / ch;
  return ks * ((ks + apm - 1) / apm);
}

// instantiated (CH, PC, KS) variants
static bool wgm_variant_ok(int ch, int pc, int ks, int jp = 0) {
  if (ks == 3 && jp == 2) return ch == 32 && pc == 64;   // stride-2 parity classes, all dY channels in one piece
  if (ks == 3) return (ch == 32 || ch == 64) && (pc == 32 || pc == 16);
  if (ks == 5) return ch == 16 && pc == 16;
  return false;
}

// pick the role / piece sizes with the fewest MMAs per voxel tile; 0 = unsupported
static int wgm_choose(int ci, int co, int ks, int* role, int* CH, int* PC) {
  int best = 0;
  for (int r = 0; r < 2; ++r) {
    const int chh = r == 0 ? ci : co, chp = r == 0 ? co : ci;
    for (int ch : {64, 32, 16}) {
      if (chh % ch != 0) continue;
      for (int pc : {32, 16}) {
        if (chp % pc != 0 || !wgm_variant_ok(ch, pc, ks)) continue;
        if (wgm_groups(ch, ks) * ks * pc > 512) continue;
        const int cost = (chh / ch) * (chp / pc) * wgm_groups(ch, ks) * (pc == 32 ? 4 : 3);  // N = ks*32 costs ~4/3 of ks*16
        if (best == 0 || cost < best) {
          best = cost;
          *role = r;
          *CH = ch;
          *PC = pc;
        }
      }
    }
  }
  return best;
}

// ks_code: 3 / 5 = cubic kernel; 1 = planar k(1,3,3), pad (0,1,1): the k3 machinery restricted to the centre depth offset
static int plan_wgm(const rehr_tensor& x, const rehr_tensor& dy, int ks_code, WgmPlan* out, int force_role = -1, int jp2 = 0) {
  WgmParams& p = out->p;
  memset(&p, 0, sizeof(p));
  const int ks = ks_code == 1 ? 3 : ks_code;
  out->planar = ks_code == 1 ? 1 : 0;
  if (x.n != dy.n || x.d != dy.d || x.h != dy.h || x.w != dy.w) return REHR_BAD_SHAPE;
  int role = 0, CH = 0, PC = 0;
  if (wgm_choose(x.c, dy.c, ks, &role, &CH, &PC) == 0) return REHR_UNSUPPORTED;
  if (force_role >= 0 && role != force_role) {  // the caller needs a fixed operand assignment: re-pick the pieces for it
    const int chh = force_role == 0 ? x.c : dy.c, chp = force_role == 0 ? dy.c : x.c;
    CH = chh % 64 == 0 ? 64 : (chh % 32 == 0 ? 32 : 0);
    PC = chp % 32 == 0 ? 32 : (chp % 16 == 0 ? 16 : 0);
    if (CH == 0 || PC == 0 || !wgm_variant_ok(CH, PC, ks)) return REHR_UNSUPPORTED;
    role = force_role;
  }
  out->JP = ks;
  if (jp2 && force_role == 0 && x.c % 32 == 0 && x.c % 64 != 0 && dy.c % 64 == 0 && wgm_variant_ok(32, 64, ks, 2) &&
      !getenv("REHR_WGM_NO_PC64")) {
    CH = 32; PC = 64; role = 0;      // only the planes q, q + 1 own accumulators (see WgmCfg): one piece covers 64 dY channels
    out->JP = 2;
  }
  p.g_mask = 0xffff;
  p.j_min = 0;
  p.j_max = ks - 1;
  if (out->planar) p.j_min = p.j_max = 1;
  const rehr_tensor& hh = role == 0 ? x : dy;
  const rehr_tensor& pp = role == 0 ? dy : x;
  if (hh.ld % 8 != 0 || pp.ld % 8 != 0) return REHR_BAD_ALIGNMENT;
  out->CH = CH;
  out->PC = PC;
  out->KS = ks;
  out->role = role;
  out->groups = wgm_groups(CH, ks);
  p.N = x.n; p.D = x.d; p.H = x.h; p.W = x.w;
  p.tiles_h = (p.H + kWTileH - 1) / kWTileH;
  p.tiles_w = (p.W + kWTileW - 1) / kWTileW;
  p.n_hs = hh.c / CH;
  p.n_ps = pp.c / PC;
  p.n_combo = p.n_hs * p.n_ps;
  const int sms = sm_count();
  if (p.n_combo > sms) return REHR_UNSUPPORTED;
  p.ctas_per_combo = sms / p.n_combo;
  const long long cols = (long long)p.N * p.tiles_h * p.tiles_w;
  // depth segments: long (less plane re-loading) but >= ~6 items per CTA for balance
  int ds = p.D;
  while (ds > 4 && cols * ((p.D + ds - 1) / ds) < 6LL * p.ctas_per_combo) ds = (ds + 1) / 2;
  p.Ds = ds;
  p.n_seg = (p.D + ds - 1) / ds;
  p.items_per_combo = (int)(cols * p.n_seg);
  if (p.items_per_combo < p.ctas_per_combo) p.ctas_per_combo = p.items_per_combo;
  // too little work to amortise the per-CTA partial dW and its reduction (measured on B200: the generic split-K kernel
  // wins at 16^3 and below, this one from 32^3 up): leave small volumes to conv_wgrad_kernel
  if (cols * p.D < 256) return REHR_UNSUPPORTED;
  const int halo_rows = (kWTileH + ks - 1) * (kWTileW + ks - 1);
  p.h_stride = ((uint32_t)(halo_rows + 16) * CH * 2 + 1023u) & ~1023u;  // + slack rows read by discarded atoms
  out->grid = p.n_combo * p.ctas_per_combo;
  const size_t pslot = (size_t)kWTileH * kWTileW * PC * 2;
  // barriers (full / empty of both rings, zero, done) and the TMEM address.  One more barrier per slot of each ring stays reserved:
  // the halo-ring depths of the tuned layer shapes were measured with a tail of this size.
  const size_t tailb = (3 * kMaxHStages + 3 * (ks + kPSpare) + 2) * 8 + 16;
  const size_t fixed = 1024 + (((size_t)(ks + kPSpare + ks - 1) * pslot + 1023) & ~size_t(1023)) + tailb;
  {
    const char* e = getenv("REHR_WGM_HSTAGES");  // development: force the halo ring depth
    const int want = e ? atoi(e) : 4;
    p.h_stages = (int)std::min<size_t>((size_t)std::max(4, std::min(want, kMaxHStages)), (smem_budget() - fixed) / p.h_stride);
    if (p.h_stages < 4) return REHR_UNSUPPORTED;
  }
  out->smem = fixed + (size_t)p.h_stages * p.h_stride;
  out->ws_bytes = (size_t)out->grid * out->groups * 128 * out->JP * PC * sizeof(float);
  return REHR_OK;
}

template <int CH, int PC, int KS, int JP = KS>
static int launch_wgm(const WgmPlan& pl, cudaStream_t stream) {
  REHR_SET_MAX_SMEM_ONCE((wgrad_march_kernel<CH, PC, KS, JP>), 227 * 1024);
  wgrad_march_kernel<CH, PC, KS, JP><<<pl.grid, kWgmThreads, pl.smem, stream>>>(pl.p);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

}  // namespace rehr

using namespace rehr;

// launch the variant + its reduction (cls_s / cls_r: parity-class tap mapping of a stride-2 conv, or null)
static int wgm_launch_kernel(const WgmPlan& pl, cudaStream_t stream) {
  const int ks = pl.KS;
  int rc = REHR_UNSUPPORTED;
  if (ks == 3 && pl.JP == 2 && pl.CH == 32 && pl.PC == 64) rc = launch_wgm<32, 64, 3, 2>(pl, stream);
  else if (ks == 3 && pl.CH == 32 && pl.PC == 32) rc = launch_wgm<32, 32, 3>(pl, stream);
  else if (ks == 3 && pl.CH == 64 && pl.PC == 32) rc = launch_wgm<64, 32, 3>(pl, stream);
  else if (ks == 3 && pl.CH == 32 && pl.PC == 16) rc = launch_wgm<32, 16, 3>(pl, stream);
  else if (ks == 3 && pl.CH == 64 && pl.PC == 16) rc = launch_wgm<64, 16, 3>(pl, stream);
  else if (ks == 5 && pl.CH == 16 && pl.PC == 16) rc = launch_wgm<16, 16, 5>(pl, stream);
  return rc;
}

// sum the partial dW of `ctas_per_combo` x n_combo consecutive CTAs starting at `ws` into dw
static int wgm_reduce(const WgmPlan& pl, const float* ws, int ctas_per_combo, int Ci, int Co, float* dw, int accumulate,
                      const int* cls_s, const int* cls_r, cudaStream_t stream) {
  const WgmParams& p = pl.p;
  const int ks = pl.KS;
  WgmReduceParams r;
  memset(&r, 0, sizeof(r));
  r.ws = ws;
  r.dw = dw;
  r.CH = pl.CH;
  r.PC = pl.PC;
  r.KS = ks;
  r.JP = pl.JP;
  r.groups = pl.groups;
  r.apm = 128 / pl.CH;
  r.parts = (ks + r.apm - 1) / r.apm;
  r.paired = (pl.CH == 64 && ks == 3) ? 1 : 0;
  r.n_hs = p.n_hs;
  r.n_ps = p.n_ps;
  r.n_combo = p.n_combo;
  r.ctas_per_combo = ctas_per_combo;
  r.role = pl.role;
  r.Ci = Ci;
  r.Co = Co;
  r.accumulate = accumulate;
  r.planar = pl.planar;
  if (cls_s) {
    for (int a = 0; a < 3; ++a) {
      r.cls_s[a] = cls_s[a];
      r.cls_r[a] = cls_r[a];
    }
  }
  if (ctas_per_combo >= 24) {
    const int blocks = p.n_hs * p.n_ps * ks * ks * ks * pl.CH;
    wgrad_march_reduce_kernel<true><<<blocks, 256, 0, stream>>>(r);
  } else {
    const int nsub = 256 / pl.PC;
    const int chb = (pl.CH + nsub - 1) / nsub;
    const int blocks = p.n_hs * p.n_ps * ks * ks * ks * chb;
    wgrad_march_reduce_kernel<false><<<blocks, 256, 0, stream>>>(r);
  }
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

static int wgm_run(const WgmPlan& pl, int Ci, int Co, float* dw, int accumulate, const int* cls_s, const int* cls_r,
                   cudaStream_t stream) {
  int rc = wgm_launch_kernel(pl, stream);
  if (rc != REHR_OK) return rc;
  return wgm_reduce(pl, pl.p.ws, pl.p.ctas_per_combo, Ci, Co, dw, accumulate, cls_s, cls_r, stream);
}

static int wgm_ks_of(const rehr_conv_desc* d) {
  if (!d) return 0;
  if (d->kd == 1 && d->kh == 3 && d->kw == 3 && d->sd == 1 && d->sh == 1 && d->sw == 1 && d->pd == 0 && d->ph == 1 && d->pw == 1) return 1;
  if (d->kd != d->kh || d->kh != d->kw || (d->kd != 3 && d->kd != 5)) return 0;
  if (d->sd != 1 || d->sh != 1 || d->sw != 1) return 0;
  const int r = (d->kd - 1) / 2;
  if (d->pd != r || d->ph != r || d->pw != r) return 0;
  return d->kd;
}

extern "C" {

int rehr_conv3d_wgrad_march_supported(const rehr_conv_desc* d, const rehr_tensor* x, const rehr_tensor* dy) {
  if (!x || !dy) return 0;
  const int ks = wgm_ks_of(d);
  if (ks == 0) return 0;
  WgmPlan pl;
  return plan_wgm(*x, *dy, ks, &pl) == REHR_OK ? 1 : 0;
}

size_t rehr_conv3d_wgrad_march_workspace(const rehr_tensor* x, const rehr_tensor* dy, int ks) {
  if (!x || !dy) return 0;
  WgmPlan pl;
  if (plan_wgm(*x, *dy, ks, &pl) != REHR_OK) return 0;
  return pl.ws_bytes;
}

// dw: f32 [cout][x->c][ks^3] (ks = 1: planar k(1,3,3) layer, dw [cout][x->c][9]); `cout` <= dy->c lets the caller pass a dy zero-padded to a multiple of 16 channels.
int rehr_conv3d_wgrad_march(const rehr_tensor* x, const rehr_tensor* dy, int ks, int cout, float* dw, int accumulate, void* ws,
                            size_t ws_bytes, rehr_stream stream_) {
  if (!x || !dy || !x->ptr || !dy->ptr || !dw || cout <= 0 || cout > dy->c) return REHR_BAD_SHAPE;
  if (dy->dtype != REHR_BF16 || x->dtype != REHR_BF16) return REHR_UNSUPPORTED;  // one MMA, one 16-bit format
  cudaStream_t stream = (cudaStream_t)stream_;
  WgmPlan pl;
  int rc = plan_wgm(*x, *dy, ks, &pl);
  if (rc != REHR_OK) return rc;
  if (!ws || ws_bytes < pl.ws_bytes) return REHR_WORKSPACE;
  WgmParams& p = pl.p;
  p.ws = reinterpret_cast<float*>(ws);
  p.err = nullptr;
  const rehr_tensor& hh = pl.role == 0 ? *x : *dy;
  const rehr_tensor& pp = pl.role == 0 ? *dy : *x;
  {
    const unsigned long long gdim[5] = {(unsigned long long)hh.c, (unsigned long long)hh.w, (unsigned long long)hh.h,
                                        (unsigned long long)hh.d, (unsigned long long)hh.n};
    const unsigned long long pitch = (unsigned long long)hh.ld * 2;
    const unsigned long long gstr[4] = {pitch, pitch * hh.w, pitch * hh.w * hh.h, pitch * hh.w * hh.h * hh.d};
    const unsigned box[5] = {(unsigned)pl.CH, (unsigned)(kWTileW + pl.KS - 1), (unsigned)(kWTileH + pl.KS - 1), 1u, 1u};
    rc = encode_tiled_bf16(&p.h_map, hh.ptr, 5, gdim, gstr, box, pl.CH * 2);
    if (rc != REHR_OK) return rc;
  }
  {
    const unsigned long long gdim[5] = {(unsigned long long)pp.c, (unsigned long long)pp.w, (unsigned long long)pp.h,
                                        (unsigned long long)pp.d, (unsigned long long)pp.n};
    const unsigned long long pitch = (unsigned long long)pp.ld * 2;
    const unsigned long long gstr[4] = {pitch, pitch * pp.w, pitch * pp.w * pp.h, pitch * pp.w * pp.h * pp.d};
    const unsigned box[5] = {(unsigned)pl.PC, (unsigned)kWTileW, (unsigned)kWTileH, 1u, 1u};
    rc = encode_tiled_bf16(&p.p_map, pp.ptr, 5, gdim, gstr, box, pl.PC * 2);
    if (rc != REHR_OK) return rc;
  }
  return wgm_run(pl, x->c, cout, dw, accumulate, nullptr, nullptr, stream);
}

// ---- weight gradient of a k3 / pad 1 conv with strides in {1, 2}: one marching pass per parity class of X -------------------
static bool wgm_s2_desc_ok(const rehr_conv_desc* d) {
  if (!d) return false;
  if (d->kd != 3 || d->kh != 3 || d->kw != 3 || d->pd != 1 || d->ph != 1 || d->pw != 1) return false;
  if ((d->sd != 1 && d->sd != 2) || (d->sh != 1 && d->sh != 2) || (d->sw != 1 && d->sw != 2)) return false;
  return d->sd * d->sh * d->sw > 1;
}

static int wgm_s2_plan(const rehr_conv_desc* d, const rehr_tensor* x, const rehr_tensor* dy, WgmPlan* pl) {
  if (!wgm_s2_desc_ok(d) || !x || !dy) return REHR_UNSUPPORTED;
  const int s[3] = {d->sd, d->sh, d->sw};
  const int in[3] = {x->d, x->h, x->w}, out[3] = {dy->d, dy->h, dy->w};
  for (int a = 0; a < 3; ++a)
    if (out[a] != (in[a] + 2 - 3) / s[a] + 1) return REHR_BAD_SHAPE;
  if (x->n != dy->n) return REHR_BAD_SHAPE;
  rehr_tensor xv = *dy;  // the iteration space is the dy grid; the halo operand is a parity class of X with X's channels
  xv.c = x->c;
  xv.ld = x->ld;
  return plan_wgm(xv, *dy, 3, pl, 0, d->sd == 2 ? 1 : 0);   // depth stride 2: no class uses the plane q - 1
}

int rehr_conv3d_wgrad_march_s2_supported(const rehr_conv_desc* d, const rehr_tensor* x, const rehr_tensor* dy) {
  WgmPlan pl;
  return wgm_s2_plan(d, x, dy, &pl) == REHR_OK ? 1 : 0;
}
size_t rehr_conv3d_wgrad_march_s2_workspace(const rehr_conv_desc* d, const rehr_tensor* x, const rehr_tensor* dy) {
  WgmPlan pl;
  if (wgm_s2_plan(d, x, dy, &pl) != REHR_OK) return 0;
  return pl.ws_bytes;
}
int rehr_conv3d_wgrad_march_s2(const rehr_conv_desc* d, const rehr_tensor* x, const rehr_tensor* dy, float* dw, int accumulate,
                               void* ws, size_t ws_bytes, rehr_stream stream_) {
  if (!x || !dy || !x->ptr || !dy->ptr || !dw) return REHR_BAD_SHAPE;
  if (dy->dtype != REHR_BF16 || x->dtype != REHR_BF16) return REHR_UNSUPPORTED;
  cudaStream_t stream = (cudaStream_t)stream_;
  WgmPlan pl;
  int rc = wgm_s2_plan(d, x, dy, &pl);
  if (rc != REHR_OK) return rc;
  if (!ws || ws_bytes < pl.ws_bytes) return REHR_WORKSPACE;
  const int s[3] = {d->sd, d->sh, d->sw};
  const int in[3] = {x->d, x->h, x->w};
  const unsigned long long pitch = (unsigned long long)x->ld * 2;  // bytes
  const unsigned long long xpw = pitch, xph = pitch * x->w, xpd = xph * x->h, xpn = xpd * x->d;
  {
    const unsigned long long gdim[5] = {(unsigned long long)dy->c, (unsigned long long)dy->w, (unsigned long long)dy->h,
                                        (unsigned long long)dy->d, (unsigned long long)dy->n};
    const unsigned long long dp = (unsigned long long)dy->ld * 2;
    const unsigned long long gstr[4] = {dp, dp * dy->w, dp * dy->w * dy->h, dp * dy->w * dy->h * dy->d};
    const unsigned box[5] = {(unsigned)pl.PC, (unsigned)kWTileW, (unsigned)kWTileH, 1u, 1u};
    rc = encode_tiled_bf16(&pl.p.p_map, dy->ptr, 5, gdim, gstr, box, pl.PC * 2);
    if (rc != REHR_OK) return rc;
  }
  pl.p.ws = reinterpret_cast<float*>(ws);
  pl.p.err = nullptr;
  // all parity classes in ONE launch: class c owns the CTAs [cls_begin[c], cls_begin[c + 1]), sized by its MMA count
  WgmParams& p = pl.p;
  int n_cls = 0, cost[8], cls_r[8][3];
  for (int rd = 0; rd < s[0]; ++rd)
    for (int rh = 0; rh < s[1]; ++rh)
      for (int rw = 0; rw < s[2]; ++rw) {
        const int r[3] = {rd, rh, rw};
        int ext[3];
        bool empty = false;
        for (int a = 0; a < 3; ++a) {
          ext[a] = (in[a] - r[a] + s[a] - 1) / s[a];
          if (ext[a] <= 0) empty = true;
        }
        if (empty) continue;
        // halo operand = class view of X: extents ext, doubled pitches, base offset r
        const unsigned long long gdim[5] = {(unsigned long long)x->c, (unsigned long long)ext[2], (unsigned long long)ext[1],
                                            (unsigned long long)ext[0], (unsigned long long)x->n};
        const unsigned long long gstr[4] = {xpw * s[2], xph * s[1], xpd * s[0], xpn};
        const unsigned box[5] = {(unsigned)pl.CH, (unsigned)(kWTileW + 2), (unsigned)(kWTileH + 2), 1u, 1u};
        const uint8_t* base = reinterpret_cast<const uint8_t*>(x->ptr) + rd * xpd + rh * xph + rw * xpw;
        rc = encode_tiled_bf16(&p.h_maps[n_cls], base, 5, gdim, gstr, box, pl.CH * 2);
        if (rc != REHR_OK) return rc;
        // offsets e needed per dim: stride 1 -> {-1, 0, 1}; stride 2: r = 0 -> {0}; r = 1 -> {-1, 0}
        int elo[3], ehi[3];
        for (int a = 0; a < 3; ++a) {
          if (s[a] == 1) { elo[a] = -1; ehi[a] = 1; }
          else if (r[a] == 0) { elo[a] = 0; ehi[a] = 0; }
          else { elo[a] = -1; ehi[a] = 0; }
        }
        // depth: e_d = 1 - j  ->  j in [1 - ehi, 1 - elo];  in-plane: offset index oh = e_h + 1, ow = e_w + 1
        p.cls_jmin[n_cls] = 1 - ehi[0];
        p.cls_jmax[n_cls] = 1 - elo[0];
        int gmask = 0;
        for (int oh = elo[1] + 1; oh <= ehi[1] + 1; ++oh)
          for (int ow = elo[2] + 1; ow <= ehi[2] + 1; ++ow) {
            const int a = oh * 3 + ow;
            gmask |= 1 << (pl.CH == 64 ? a / 2 : oh);
          }
        p.cls_gmask[n_cls] = gmask;
        cost[n_cls] = __builtin_popcount(gmask);
        for (int a = 0; a < 3; ++a) cls_r[n_cls][a] = r[a];
        ++n_cls;
      }
  if (n_cls == 0) return REHR_OK;
  // CTA shares proportional to the MMA groups a class issues per plane; multiples of n_combo, at least one combo set each
  const int budget = pl.grid / p.n_combo;  // combo sets available (<= SMs)
  if (budget < n_cls) return REHR_UNSUPPORTED;
  int total_cost = 0, share[8], used = 0;
  for (int c = 0; c < n_cls; ++c) total_cost += cost[c];
  for (int c = 0; c < n_cls; ++c) {
    share[c] = std::max(1, (int)((long long)budget * cost[c] / total_cost));
    share[c] = std::min(share[c], p.items_per_combo);
    used += share[c];
  }
  for (int c = 0; used > budget; c = (c + 1) % n_cls)
    if (share[c] > 1) { --share[c]; --used; }
  p.n_cls = n_cls;
  p.cls_begin[0] = 0;
  for (int c = 0; c < n_cls; ++c) p.cls_begin[c + 1] = p.cls_begin[c] + share[c] * p.n_combo;
  pl.grid = p.cls_begin[n_cls];
  rc = wgm_launch_kernel(pl, stream);
  if (rc != REHR_OK) return rc;
  const size_t per_cta = (size_t)pl.groups * 128 * pl.JP * pl.PC;
  const int cs[3] = {s[0], s[1], s[2]};
  for (int c = 0; c < n_cls; ++c) {
    rc = wgm_reduce(pl, p.ws + (size_t)p.cls_begin[c] * per_cta, share[c], x->c, dy->c, dw, accumulate, cs, cls_r[c], stream);
    if (rc != REHR_OK) return rc;
  }
  return REHR_OK;
}

}  // extern "C"
