// Fused reduction kernels for the stage-2 and SR-stage losses (SURVEY.md 8(f) row 4: "the losses as fused CE+Dice reductions"), all HBM-bound
// single passes over fp32 NCDHW tensors exactly as the caller holds them (no layout change):
//
//   * segmentation loss sums   <- DC_and_weighted_CE_loss, utils/seg_utils.py:305-353 (RobustCrossEntropyLoss :289-303 and the
//                                 nnunetv2 MemoryEfficientSoftDiceLoss): per sample the weighted cross-entropy sum and the
//                                 per-class soft-Dice sums (intersection, prediction mass, label count) from ONE read of the logits;
//   * channel-cosine sums      <- cosine_distance_loss, models/seg_model.py:60-78: per (sample, channel) sums over the voxels of
//                                 the channel-normalised maps (a.b, a.a, b.b);
//   * plane max-pool           <- CriterionPairWiseforWholeFeatAfterPool, models/seg_model.py:95-113: per (sample, channel, slice)
//                                 max over non-overlapping in-plane windows (ceil mode) with the arg-max for the backward scatter;
//   * SR-stage loss sums       <- the loss statements of train_sr, train_all.py:124-133 (L1, the UASR terms, BCEDiceLoss): the
//                                 voxel sums of all of them from ONE read of the network output, the target window and u.
//
// Each forward kernel only produces the SUMS; the few scalars of the actual loss (Dice ratio, 1 - cos, Gram matrices) are then
// ordinary autograd ops on tiny tensors in rehrseg_b200/loss_ops.py, and each backward kernel turns the gradients of those sums
// into the dense gradient in one more pass.  Deterministic: per-warp slots / per-block partials, fixed summation order.
#include "engine.h"

#include <algorithm>
#include <cfloat>
#include <cstdint>

namespace rehr {

static constexpr int kLossMaxClasses = 8;
static constexpr int kSrMaxChannels = 4;   // SR-stage output channels (the reference has 2); more spill the unrolled accumulators

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------------------------------
// segmentation loss sums.  logits [B][C][V] f32, target [B][V] f32 (class index), weight [V] f32 or null (the CE map of EVERY
// sample is multiplied by it: the reference's [B,D,H,W] x [B,1,D,H,W] broadcast makes the weight sum_b' uncertainty[b'] / B).
// partial [B][blocks][1 + 3*C]: 0 = sum_v w*ce, then per class: sum p*[y=c], sum p, sum [y=c].
// ------------------------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(256) seg_loss_sums_kernel(const float* __restrict__ logits, const float* __restrict__ target,
                                                            const float* __restrict__ weight, long long V, float* __restrict__ partial) {
  constexpr int K = 1 + 3 * C;
  __shared__ float slot[8][K];
  const int b = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* lg = logits + (long long)b * C * V;
  const float* tg = target + (long long)b * V;
  float acc[K];
#pragma unroll
  for (int i = 0; i < K; ++i) acc[i] = 0.f;
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < V; v += (long long)gridDim.x * blockDim.x) {
    float z[C];
#pragma unroll
    for (int c = 0; c < C; ++c) z[c] = __ldcs(lg + (long long)c * V + v);
    const int y = (int)__ldcs(tg + v);
    const float w = weight ? __ldg(weight + v) : 1.f;
    float m = z[0];
#pragma unroll
    for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
    float e[C], s = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      e[c] = __expf(z[c] - m);
      s += e[c];
    }
    const float inv = 1.f / s, lse = m + __logf(s);
    float zy = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const float p = e[c] * inv;
      const bool hit = (y == c);
      zy = hit ? z[c] : zy;
      acc[1 + 3 * c] += hit ? p : 0.f;
      acc[2 + 3 * c] += p;
      acc[3 + 3 * c] += hit ? 1.f : 0.f;
    }
    acc[0] += w * (lse - zy);
  }
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const float t = warp_sum(acc[i]);
    if (lane == 0) slot[warp][i] = t;
  }
  __syncthreads();
  if (threadIdx.x < K) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += slot[w][threadIdx.x];
    partial[((long long)b * gridDim.x + blockIdx.x) * K + threadIdx.x] = t;
  }
}

// dlogits[b][k][v] = g_ce[b] * w[v] * (p_k - [y=k]) + p_k * (h_k - sum_c h_c p_c),  h_c = g_int[b][c] * [y=c] + g_pred[b][c]
template <int C>
__global__ void __launch_bounds__(256) seg_loss_bwd_kernel(const float* __restrict__ logits, const float* __restrict__ target,
                                                           const float* __restrict__ weight, long long V, const float* __restrict__ g_ce,
                                                           const float* __restrict__ g_int, const float* __restrict__ g_pred,
                                                           float* __restrict__ dlogits) {
  const int b = blockIdx.y;
  const float* lg = logits + (long long)b * C * V;
  const float* tg = target + (long long)b * V;
  float* dl = dlogits + (long long)b * C * V;
  const float gce = g_ce[b];
  float gi[C], gp[C];
#pragma unroll
  for (int c = 0; c < C; ++c) {
    gi[c] = g_int[b * C + c];
    gp[c] = g_pred[b * C + c];
  }
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < V; v += (long long)gridDim.x * blockDim.x) {
    float z[C];
#pragma unroll
    for (int c = 0; c < C; ++c) z[c] = __ldcs(lg + (long long)c * V + v);
    const int y = (int)__ldcs(tg + v);
    const float w = (weight ? __ldg(weight + v) : 1.f) * gce;
    float m = z[0];
#pragma unroll
    for (int c = 1; c < C; ++c) m = fmaxf(m, z[c]);
    float p[C], s = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      p[c] = __expf(z[c] - m);
      s += p[c];
    }
    const float inv = 1.f / s;
    float hp = 0.f, h[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
      p[c] *= inv;
      h[c] = gp[c] + (y == c ? gi[c] : 0.f);
      hp = fmaf(h[c], p[c], hp);
    }
#pragma unroll
    for (int c = 0; c < C; ++c) __stcs(dl + (long long)c * V + v, w * (p[c] - (y == c ? 1.f : 0.f)) + p[c] * (h[c] - hp));
  }
}

// ------------------------------------------------------------------------------------------------------------------
// channel-cosine sums.  a, b [B][C][V] f32.  ahat = a / max(||a[:, v]||_2, 1e-12) (F.normalize over the channel axis), same for b;
// partial [B][blocks][3][C]: sum_v ahat*bhat, sum_v ahat^2, sum_v bhat^2.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cosine_sums_kernel(const float* __restrict__ a, const float* __restrict__ b, int C, long long V,
                                                          float* __restrict__ partial) {
  extern __shared__ float slot[];  // [8 warps][3][C]
  const int n = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* pa = a + (long long)n * C * V;
  const float* pb = b + (long long)n * C * V;
  for (int i = threadIdx.x; i < 8 * 3 * C; i += blockDim.x) slot[i] = 0.f;
  __syncthreads();
  float* mine = slot + warp * 3 * C;
  const long long stride = (long long)gridDim.x * blockDim.x;
  // whole warps iterate together (the tail lanes contribute zeros) so that the shuffles stay convergent
  for (long long v0 = blockIdx.x * (long long)blockDim.x + warp * 32; v0 < V; v0 += stride) {
    const long long v = v0 + lane;
    const bool ok = v < V;
    float na = 0.f, nb = 0.f;
#pragma unroll 8
    for (int c = 0; c < C; ++c) {
      const float x = ok ? __ldg(pa + (long long)c * V + v) : 0.f;
      const float y = ok ? __ldg(pb + (long long)c * V + v) : 0.f;
      na = fmaf(x, x, na);
      nb = fmaf(y, y, nb);
    }
    const float ia = 1.f / fmaxf(sqrtf(na), 1e-12f), ib = 1.f / fmaxf(sqrtf(nb), 1e-12f);
    for (int c = 0; c < C; ++c) {
      const float x = (ok ? __ldg(pa + (long long)c * V + v) : 0.f) * ia;   // second read: L1 / L2 hit
      const float y = (ok ? __ldg(pb + (long long)c * V + v) : 0.f) * ib;
      const float s0 = warp_sum(x * y), s1 = warp_sum(x * x), s2 = warp_sum(y * y);
      if (lane == 0) {
        mine[c] += s0;
        mine[C + c] += s1;
        mine[2 * C + c] += s2;
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * C; i += blockDim.x) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += slot[w * 3 * C + i];
    partial[((long long)n * gridDim.x + blockIdx.x) * 3 * C + i] = t;
  }
}

// da[c][v] = ia * (G[c][v] - ahat[c][v] * sum_c' G[c'][v] ahat[c'][v]),  G = gP[c] * bhat + 2 gQ[c] * ahat   (b has no gradient)
__global__ void __launch_bounds__(256) cosine_sums_bwd_kernel(const float* __restrict__ a, const float* __restrict__ b, int C, long long V,
                                                              const float* __restrict__ gP, const float* __restrict__ gQ,
                                                              float* __restrict__ da) {
  extern __shared__ float sg[];  // [2][C]
  const int n = blockIdx.y;
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    sg[i] = gP[n * C + i];
    sg[C + i] = 2.f * gQ[n * C + i];
  }
  __syncthreads();
  const float* pa = a + (long long)n * C * V;
  const float* pb = b + (long long)n * C * V;
  float* pd = da + (long long)n * C * V;
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < V; v += (long long)gridDim.x * blockDim.x) {
    float na = 0.f, nb = 0.f;
#pragma unroll 8
    for (int c = 0; c < C; ++c) {
      const float x = __ldg(pa + (long long)c * V + v), y = __ldg(pb + (long long)c * V + v);
      na = fmaf(x, x, na);
      nb = fmaf(y, y, nb);
    }
    const float ra = sqrtf(na);
    const float ia = 1.f / fmaxf(ra, 1e-12f), ib = 1.f / fmaxf(sqrtf(nb), 1e-12f);
    float dot = 0.f;
    for (int c = 0; c < C; ++c) {
      const float x = __ldg(pa + (long long)c * V + v) * ia, y = __ldg(pb + (long long)c * V + v) * ib;
      dot = fmaf(sg[c] * y + sg[C + c] * x, x, dot);
    }
    if (ra <= 1e-12f) dot = 0.f;  // clamped norm: ahat = a / eps is linear in a
    for (int c = 0; c < C; ++c) {
      const float x = __ldg(pa + (long long)c * V + v) * ia, y = __ldg(pb + (long long)c * V + v) * ib;
      __stcs(pd + (long long)c * V + v, ia * (sg[c] * y + sg[C + c] * x - x * dot));
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// plane max-pool.  x [N][C][S][H][W] f32; windows ph x pw, stride = window, ceil mode (the last window may be partial).
// out [N][S][C][OH][OW] f32 (= the reference's '(b s) c h w' pooled tensor), idx same shape int32 (offset inside the H*W plane of the
// FIRST maximum in row-major order, as ATen's max_pool2d picks it).  One CTA per (n, c, s) plane.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) plane_maxpool_kernel(const float* __restrict__ x, int C, int S, int H, int W, int ph, int pw, int OH,
                                                            int OW, float* __restrict__ out, int* __restrict__ idx) {
  __shared__ float sv[8];
  __shared__ int si[8];
  const int plane = blockIdx.x;  // (n*C + c)*S + s
  const int s = plane % S, c = (plane / S) % C, n = plane / (S * C);
  const float* p = x + (long long)plane * H * W;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int win = 0; win < OH * OW; ++win) {
    const int h0 = (win / OW) * ph, w0 = (win % OW) * pw;
    const int hh = min(ph, H - h0), ww = min(pw, W - w0);
    float best = -FLT_MAX;
    int bi = 0x7fffffff;
    for (int i = threadIdx.x; i < hh * ww; i += blockDim.x) {  // increasing offsets per thread: first maximum kept by '>'
      const int off = (h0 + i / ww) * W + w0 + i % ww;
      const float v = __ldg(p + off);
      if (v > best || (v != v && bi == 0x7fffffff)) {
        best = v;
        bi = off;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > best || (ov == best && oi < bi)) {
        best = ov;
        bi = oi;
      }
    }
    __syncthreads();
    if (lane == 0) {
      sv[warp] = best;
      si[warp] = bi;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
      for (int w = 1; w < 8; ++w)
        if (sv[w] > best || (sv[w] == best && si[w] < bi)) {
          best = sv[w];
          bi = si[w];
        }
      const long long o = (((long long)n * S + s) * C + c) * (OH * OW) + win;
      out[o] = best;
      idx[o] = bi;
    }
  }
}

// dx (zero-filled by the caller) [N][C][S][H][W]: dx[plane][idx] = g  (windows do not overlap: one writer per element)
__global__ void plane_maxpool_bwd_kernel(const float* __restrict__ g, const int* __restrict__ idx, int C, int S, int HW, int OHW,
                                         long long total, float* __restrict__ dx) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int win = (int)(i % OHW);
  long long r = i / OHW;
  const int c = (int)(r % C);
  r /= C;
  const int s = (int)(r % S);
  const long long n = r / S;
  (void)win;
  dx[((n * C + c) * S + s) * HW + idx[i]] = g[i];
}

// ------------------------------------------------------------------------------------------------------------------
// SR-stage loss sums <- train_all.py:124-133: L1Loss on channel 0, the UASR terms :126-129 and BCEDiceLoss (utils/seg_utils.py:
// 821-886) on channels 1..C-1, from ONE read of the network output, the target and the uncertainty.
// hat [B][C][S][HW] f32 contiguous; target [B][C][S][HW] with contiguous H*W planes and the given batch / channel / depth strides
// (the depth window of patches_hr is read in place); u [B][1][S][HW] or null.  e = hat_0 - t_0, p = sigmoid(hat_c), y = t_c.
// partial [blocks][3 + 4 (C-1)]: sum |e|, sum |e|/u + log u, sum |u - |e||, then per segmentation channel sum bce, sum p*y,
// sum p^2, sum y^2.  One item = four voxels of one plane: 16-byte accesses when every plane start is aligned (VEC), masked
// scalars otherwise (ragged H*W, odd strides).
// ------------------------------------------------------------------------------------------------------------------
struct SrLossView {
  const float* hat;
  const float* target;
  const float* u;
  long long tb, tc, ts;  // target strides (elements)
  int S, HW;
  long long items;       // B * S * ceil(HW / 4)
};

template <bool VEC>
__device__ __forceinline__ void sr_ld4(const float* p, int n, bool last_use, float (&v)[4]) {
  if (VEC) {
    const float4 t = last_use ? __ldcs(reinterpret_cast<const float4*>(p)) : __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = k < n ? (last_use ? __ldcs(p + k) : __ldg(p + k)) : 0.f;
  }
}

template <bool VEC>
__device__ __forceinline__ void sr_st4(float* p, int n, const float (&v)[4]) {
  if (VEC) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (k < n) p[k] = v[k];
  }
}

// sigmoid(x) and 1 - sigmoid(x), each without cancellation; ex = exp(-|x|) is returned for the BCE's log1p
__device__ __forceinline__ void sr_sigmoid(float x, float& p, float& q, float& ex) {
  ex = expf(-fabsf(x));
  const float r = 1.f / (1.f + ex);
  p = x >= 0.f ? r : ex * r;
  q = x >= 0.f ? ex * r : r;
}

__device__ __forceinline__ float sr_sign(float v) { return v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f); }  // sign(0) = 0, as torch

// item i -> (plane = b*S + s, first voxel of the item inside the plane, valid voxels)
__device__ __forceinline__ void sr_item(const SrLossView& a, long long i, long long& plane, long long& b, int& s, int& off, int& n) {
  const int vpp = (a.HW + 3) >> 2;
  plane = i / vpp;
  off = (int)(i - plane * vpp) * 4;
  n = min(4, a.HW - off);
  b = plane / a.S;
  s = (int)(plane - b * a.S);
}

template <int C, bool VEC>
__global__ void __launch_bounds__(256) sr_loss_sums_kernel(const SrLossView a, float* __restrict__ partial) {
  constexpr int K = 3 + 4 * (C - 1);
  __shared__ float slot[8][K];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long cstride = (long long)a.S * a.HW;
  float acc[K];
#pragma unroll
  for (int i = 0; i < K; ++i) acc[i] = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.items; i += (long long)gridDim.x * blockDim.x) {
    long long plane, b;
    int s, off, n;
    sr_item(a, i, plane, b, s, off, n);
    const float* h = a.hat + (b * C * a.S + s) * (long long)a.HW + off;
    const float* t = a.target + b * a.tb + s * a.ts + off;
    float hv[4], tv[4];
    sr_ld4<VEC>(h, n, false, hv);
    sr_ld4<VEC>(t, n, false, tv);
    if (a.u) {
      float uv[4];
      sr_ld4<VEC>(a.u + plane * a.HW + off, n, false, uv);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (VEC || k < n) {
          const float ae = fabsf(hv[k] - tv[k]);
          acc[0] += ae;
          acc[1] += ae / uv[k] + logf(uv[k]);
          acc[2] += fabsf(uv[k] - ae);
        }
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (VEC || k < n) acc[0] += fabsf(hv[k] - tv[k]);
    }
#pragma unroll
    for (int c = 1; c < C; ++c) {
      sr_ld4<VEC>(h + c * cstride, n, false, hv);
      sr_ld4<VEC>(t + c * a.tc, n, false, tv);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (VEC || k < n) {
          const float x = hv[k], y = tv[k];
          float p, q, ex;
          sr_sigmoid(x, p, q, ex);
          acc[4 * c - 1] += (1.f - y) * x + fmaxf(-x, 0.f) + log1pf(ex);
          acc[4 * c] += p * y;
          acc[4 * c + 1] += p * p;
          acc[4 * c + 2] += y * y;
        }
    }
  }
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const float t = warp_sum(acc[i]);
    if (lane == 0) slot[warp][i] = t;
  }
  __syncthreads();
  if (threadIdx.x < K) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += slot[w][threadIdx.x];
    partial[(long long)blockIdx.x * K + threadIdx.x] = t;
  }
}

// g [3 + 4 (C-1)]: the gradients of the sums, in the order of the partials (the sum y^2 entries are ignored).
//   d hat_0 = sign(e) (g_abs + g_uasr / u)                    (the sum |u - |e|| has no hat gradient: the error map is detached)
//   d u     = g_uasr / u (1 - |e| / u) + g_l1u sign(u - |e|)
//   d hat_c = g_bce (p - y) + (g_py y + 2 g_pp p) p (1 - p)
template <int C, bool VEC>
__global__ void __launch_bounds__(256) sr_loss_bwd_kernel(const SrLossView a, const float* __restrict__ g, float* __restrict__ d_hat,
                                                          float* __restrict__ d_u) {
  const float g_abs = g[0], g_uasr = g[1], g_l1u = g[2];
  float gb[C], gy[C], gp[C];
#pragma unroll
  for (int c = 1; c < C; ++c) {
    gb[c] = g[4 * c - 1];
    gy[c] = g[4 * c];
    gp[c] = 2.f * g[4 * c + 1];
  }
  const long long cstride = (long long)a.S * a.HW;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.items; i += (long long)gridDim.x * blockDim.x) {
    long long plane, b;
    int s, off, n;
    sr_item(a, i, plane, b, s, off, n);
    const long long ho = (b * C * a.S + s) * (long long)a.HW + off;
    const float* t = a.target + b * a.tb + s * a.ts + off;
    float hv[4], tv[4], dv[4];
    sr_ld4<VEC>(a.hat + ho, n, true, hv);
    sr_ld4<VEC>(t, n, true, tv);
    if (a.u) {
      float uv[4], du[4];
      sr_ld4<VEC>(a.u + plane * a.HW + off, n, true, uv);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float e = hv[k] - tv[k], ae = fabsf(e), gu = g_uasr / uv[k];
        dv[k] = sr_sign(e) * (g_abs + gu);
        du[k] = gu * (1.f - ae / uv[k]) + g_l1u * sr_sign(uv[k] - ae);
      }
      sr_st4<VEC>(d_u + plane * a.HW + off, n, du);
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) dv[k] = sr_sign(hv[k] - tv[k]) * g_abs;
    }
    sr_st4<VEC>(d_hat + ho, n, dv);
#pragma unroll
    for (int c = 1; c < C; ++c) {
      sr_ld4<VEC>(a.hat + ho + c * cstride, n, true, hv);
      sr_ld4<VEC>(t + c * a.tc, n, true, tv);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float y = tv[k];
        float p, q, ex;
        sr_sigmoid(hv[k], p, q, ex);
        dv[k] = gb[c] * ((1.f - y) * p - y * q) + (gy[c] * y + gp[c] * p) * (p * q);   // p - y, exact at saturated logits
      }
      sr_st4<VEC>(d_hat + ho + c * cstride, n, dv);
    }
  }
}

static int loss_blocks(long long V) { return (int)std::max<long long>(1, std::min<long long>((V + 255) / 256, (long long)sm_count() * 4)); }

static bool sr_view(const float* hat, const float* target, const float* u, int B, int C, int S, int HW, long long tb, long long tc,
                    long long ts, SrLossView& a) {
  if (!hat || !target || B <= 0 || C < 2 || S <= 0 || HW <= 0) return false;
  a = SrLossView{hat, target, u, tb, tc, ts, S, HW, (long long)B * S * ((HW + 3) / 4)};
  return true;
}

static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

// every plane start of every tensor is 16-byte aligned
static bool sr_vec(const SrLossView& a, const float* d_hat, const float* d_u) {
  return a.HW % 4 == 0 && a.tb % 4 == 0 && a.tc % 4 == 0 && a.ts % 4 == 0 && aligned16(a.hat) && aligned16(a.target) &&
         aligned16(a.u) && aligned16(d_hat) && aligned16(d_u);
}

}  // namespace rehr

using namespace rehr;

extern "C" {

int rehr_loss_blocks(long long voxels) { return voxels > 0 ? loss_blocks(voxels) : 0; }

int rehr_seg_loss_sums(const float* logits, const float* target, const float* weight, int B, int C, long long V, float* partial,
                       rehr_stream stream) {
  if (!logits || !target || !partial || B <= 0 || V <= 0) return REHR_BAD_SHAPE;
  if (C < 2 || C > kLossMaxClasses) return REHR_UNSUPPORTED;
  const dim3 grid((unsigned)loss_blocks(V), (unsigned)B);
  switch (C) {
#define REHR_SEG_CASE(N) \
  case N: seg_loss_sums_kernel<N><<<grid, 256, 0, (cudaStream_t)stream>>>(logits, target, weight, V, partial); break;
    REHR_SEG_CASE(2) REHR_SEG_CASE(3) REHR_SEG_CASE(4) REHR_SEG_CASE(5) REHR_SEG_CASE(6) REHR_SEG_CASE(7) REHR_SEG_CASE(8)
#undef REHR_SEG_CASE
  }
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_seg_loss_bwd(const float* logits, const float* target, const float* weight, int B, int C, long long V, const float* g_ce,
                      const float* g_int, const float* g_pred, float* dlogits, rehr_stream stream) {
  if (!logits || !target || !g_ce || !g_int || !g_pred || !dlogits || B <= 0 || V <= 0) return REHR_BAD_SHAPE;
  if (C < 2 || C > kLossMaxClasses) return REHR_UNSUPPORTED;
  const dim3 grid((unsigned)loss_blocks(V), (unsigned)B);
  switch (C) {
#define REHR_SEG_CASE(N) \
  case N: seg_loss_bwd_kernel<N><<<grid, 256, 0, (cudaStream_t)stream>>>(logits, target, weight, V, g_ce, g_int, g_pred, dlogits); break;
    REHR_SEG_CASE(2) REHR_SEG_CASE(3) REHR_SEG_CASE(4) REHR_SEG_CASE(5) REHR_SEG_CASE(6) REHR_SEG_CASE(7) REHR_SEG_CASE(8)
#undef REHR_SEG_CASE
  }
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

#define REHR_SR_DISPATCH(LAUNCH)                                                                                        \
  switch (C) {                                                                                                           \
    case 2: LAUNCH(2); break;                                                                                            \
    case 3: LAUNCH(3); break;                                                                                            \
    case 4: LAUNCH(4); break;                                                                                            \
  }

int rehr_sr_loss_sums(const float* hat, const float* target, const float* u, int B, int C, int S, int HW, long long t_batch,
                      long long t_channel, long long t_depth, float* partial, rehr_stream stream) {
  SrLossView a;
  if (!partial || !sr_view(hat, target, u, B, C, S, HW, t_batch, t_channel, t_depth, a)) return REHR_BAD_SHAPE;
  if (C > kSrMaxChannels) return REHR_UNSUPPORTED;
  const unsigned grid = (unsigned)loss_blocks((long long)B * S * HW);
  const bool vec = sr_vec(a, nullptr, nullptr);
#define REHR_SR_SUMS(N)                                                                  \
  if (vec) sr_loss_sums_kernel<N, true><<<grid, 256, 0, (cudaStream_t)stream>>>(a, partial); \
  else sr_loss_sums_kernel<N, false><<<grid, 256, 0, (cudaStream_t)stream>>>(a, partial)
  REHR_SR_DISPATCH(REHR_SR_SUMS)
#undef REHR_SR_SUMS
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_sr_loss_bwd(const float* hat, const float* target, const float* u, int B, int C, int S, int HW, long long t_batch,
                     long long t_channel, long long t_depth, const float* g, float* d_hat, float* d_u, rehr_stream stream) {
  SrLossView a;
  if (!g || !d_hat || (u != nullptr) != (d_u != nullptr) || !sr_view(hat, target, u, B, C, S, HW, t_batch, t_channel, t_depth, a))
    return REHR_BAD_SHAPE;
  if (C > kSrMaxChannels) return REHR_UNSUPPORTED;
  const unsigned grid = (unsigned)loss_blocks((long long)B * S * HW);
  const bool vec = sr_vec(a, d_hat, d_u);
#define REHR_SR_BWD(N)                                                                                \
  if (vec) sr_loss_bwd_kernel<N, true><<<grid, 256, 0, (cudaStream_t)stream>>>(a, g, d_hat, d_u);   \
  else sr_loss_bwd_kernel<N, false><<<grid, 256, 0, (cudaStream_t)stream>>>(a, g, d_hat, d_u)
  REHR_SR_DISPATCH(REHR_SR_BWD)
#undef REHR_SR_BWD
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}
#undef REHR_SR_DISPATCH

int rehr_cosine_sums(const float* a, const float* b, int B, int C, long long V, float* partial, rehr_stream stream) {
  if (!a || !b || !partial || B <= 0 || C <= 0 || V <= 0) return REHR_BAD_SHAPE;
  if (C > 512) return REHR_UNSUPPORTED;
  const dim3 grid((unsigned)loss_blocks(V), (unsigned)B);
  cosine_sums_kernel<<<grid, 256, (size_t)8 * 3 * C * sizeof(float), (cudaStream_t)stream>>>(a, b, C, V, partial);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_cosine_sums_bwd(const float* a, const float* b, int B, int C, long long V, const float* g_ab, const float* g_aa, float* da,
                         rehr_stream stream) {
  if (!a || !b || !g_ab || !g_aa || !da || B <= 0 || C <= 0 || V <= 0) return REHR_BAD_SHAPE;
  if (C > 512) return REHR_UNSUPPORTED;
  const dim3 grid((unsigned)loss_blocks(V), (unsigned)B);
  cosine_sums_bwd_kernel<<<grid, 256, (size_t)2 * C * sizeof(float), (cudaStream_t)stream>>>(a, b, C, V, g_ab, g_aa, da);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_plane_maxpool(const float* x, int N, int C, int S, int H, int W, int ph, int pw, float* out, int* idx, rehr_stream stream) {
  if (!x || !out || !idx || N <= 0 || C <= 0 || S <= 0 || H <= 0 || W <= 0 || ph <= 0 || pw <= 0) return REHR_BAD_SHAPE;
  const int OH = (H + ph - 1) / ph, OW = (W + pw - 1) / pw;
  const long long planes = (long long)N * C * S;
  if (planes > 0x7fffffffLL) return REHR_UNSUPPORTED;
  plane_maxpool_kernel<<<(unsigned)planes, 256, 0, (cudaStream_t)stream>>>(x, C, S, H, W, ph, pw, OH, OW, out, idx);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

int rehr_plane_maxpool_bwd(const float* g, const int* idx, int N, int C, int S, int H, int W, int ph, int pw, float* dx_zeroed,
                           rehr_stream stream) {
  if (!g || !idx || !dx_zeroed || N <= 0 || C <= 0 || S <= 0) return REHR_BAD_SHAPE;
  const int OH = (H + ph - 1) / ph, OW = (W + pw - 1) / pw;
  const long long total = (long long)N * S * C * OH * OW;
  plane_maxpool_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(g, idx, C, S, H * W, OH * OW, total,
                                                                                              dx_zeroed);
  REHR_CHECK_LAUNCH();
  return REHR_OK;
}

}  // extern "C"
